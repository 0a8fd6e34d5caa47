// Beam expansion without host synchronisation: joint (word, gate) top-k per caption over
// cur_beam x (k word candidates) x (2 gates), sticky EOS masks, back-pointer history, beam-state
// reorder, and the final sort + back-track.
// Reference: models/CaptioningModel.py:116-195 (beam_search), :197-294 (beam_search_v),
// :78-114 (_select_beam).  Statics are never copied per beam (SURVEY.md §2.1 k15): rows index
// them by caption = row / beam.
#include <cooperative_groups.h>
#include <cooperative_groups/reduce.h>
#include <cuda_fp16.h>
#include <float.h>
#include <math.h>

#include "common.cuh"
#include "vocab_head.cuh"

namespace vsr {

namespace {

// log-prob of vocabulary entry `word` in row `row` as returned by the step (post verb forcing)
__device__ __forceinline__ float row_logp(const float* logits, int ld, const float* row_max,
                                          const float* row_lsum, const int32_t* forced, int row, int word) {
  const int f = forced[row];
  if (f >= 0) return word == f ? 0.f : -1e6f;
  return (logits[(size_t)row * ld + word] - row_max[row]) - row_lsum[row];
}

struct BeamArgs {
  int t, b, cur, k, V;
  int64_t eos0, eos1;
  const float* logits; int ld;
  const float* row_max; const float* row_lsum; const int32_t* forced; const int32_t* cand;
  const float* gate_lp;
  const float* seq_lp; float* seq_lp_n;
  float *m0, *m1, *m0n, *m1n;
  const int32_t *prev_word, *prev_gate;            // previous step's picks per current slot (t > 0)
  int32_t *sel_beam, *sel_word, *sel_gate;        // this step's picks (double-buffered against prev_*)
  int32_t *hist_parent, *hist_word, *hist_gate;    // [T][b][k] slices for step t
  float *hist_score, *hist_lpw, *hist_lpg;
  const int32_t *f_beam, *f_word, *f_gate;        // forced selections for step t or null
};

constexpr int MAXC = 2 * VSR_MAX_BEAM * VSR_MAX_BEAM;  // 128 candidates per caption

struct BeamSmem {
  float seq[VSR_MAX_BEAM], m0[VSR_MAX_BEAM], m1[VSR_MAX_BEAM], ps[VSR_MAX_BEAM];
  int full[VSR_MAX_BEAM], pb[VSR_MAX_BEAM], pw[VSR_MAX_BEAM], pg[VSR_MAX_BEAM];
};

// selection for caption c by one warp; leaves the picks (parent, word, gate) in sh.pb / pw / pg
__device__ __forceinline__ void beam_select_warp(const BeamArgs& a, BeamSmem& sh, int c, int lane, bool write) {
  const int k = a.k, cur = a.cur;
  float* s_seq = sh.seq; float* s_m0 = sh.m0; float* s_m1 = sh.m1; float* s_ps = sh.ps;
  int* s_full = sh.full; int* s_pb = sh.pb; int* s_pw = sh.pw; int* s_pg = sh.pg;

  if (lane < cur) {
    float m0 = 1.f, m1 = 1.f, seq = 0.f;
    if (a.t > 0) {
      // sticky masks: a head's mask drops to 0 once the slot's previous token was its EOS (:143-144)
      seq = a.seq_lp[c * k + lane];
      m0 = a.m0[c * k + lane] * ((int64_t)a.prev_word[c * k + lane] != a.eos0 ? 1.f : 0.f);
      m1 = a.m1[c * k + lane] * ((int64_t)a.prev_gate[c * k + lane] != a.eos1 ? 1.f : 0.f);
    }
    s_seq[lane] = seq; s_m0[lane] = m0; s_m1[lane] = m1;
    s_full[lane] = (a.t == 0) ? 1 : (fminf(fmaxf(m0 + m1, 0.f), 1.f) != 0.f);
  }
  __syncwarp();

  if (a.f_beam == nullptr) {
    // candidates: idx = (parent j, i-th word candidate, gate g); lane owns idx = lane + 32*q
    float cs[MAXC / 32]; int cf[MAXC / 32]; bool used[MAXC / 32];
    const int ncand = cur * k * 2;
#pragma unroll
    for (int q = 0; q < MAXC / 32; ++q) {
      const int idx = lane + 32 * q;
      cs[q] = -INFINITY; cf[q] = 0x7fffffff; used[q] = true;
      if (idx < ncand) {
        const int j = idx / (2 * k), i = (idx >> 1) % k, g = idx & 1;
        const int row = c * cur + j;
        int word; float sc;
        if (s_full[j]) {
          word = a.cand[row * VSR_MAX_BEAM + i];
          const float wl = row_logp(a.logits, a.ld, a.row_max, a.row_lsum, a.forced, row, word);
          sc = __fadd_rn(s_seq[j], __fadd_rn(wl, a.gate_lp[row * 2 + g]));   // seq + (word + gate), :139
        } else {
          // frozen beam: old score at word 0 (both gates), -999 elsewhere (:146-150)
          word = i;
          sc = (i == 0) ? s_seq[j] : -999.f;
        }
        cs[q] = sc; cf[q] = j * 2 * a.V + word * 2 + g; used[q] = false;
      }
    }
    for (int sel = 0; sel < k; ++sel) {
      float bv = -INFINITY; int bf = 0x7fffffff;
#pragma unroll
      for (int q = 0; q < MAXC / 32; ++q)
        if (!used[q] && before(cs[q], cf[q], bv, bf)) { bv = cs[q]; bf = cf[q]; }
      {   // warp arg-best in (score desc, flat index asc) order: two redux.sync + one broadcast
        const unsigned u = __float_as_uint(bv);
        const unsigned key = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
        const unsigned kbest = __reduce_max_sync(0xffffffffu, key);
        const int fbest = (int)__reduce_min_sync(0xffffffffu, key == kbest ? (unsigned)bf : 0xffffffffu);
        const unsigned owner = __ballot_sync(0xffffffffu, key == kbest && bf == fbest);
        bv = __shfl_sync(0xffffffffu, bv, __ffs(owner) - 1);
        bf = fbest;
      }
#pragma unroll
      for (int q = 0; q < MAXC / 32; ++q) if (cf[q] == bf) used[q] = true;
      if (lane == 0) {
        const int j = bf / (2 * a.V), rem = bf - j * 2 * a.V;
        s_pb[sel] = j; s_pw[sel] = rem >> 1; s_pg[sel] = rem & 1; s_ps[sel] = bv;
      }
    }
  } else if (lane < k) {
    // trajectory replay: take the given selection, score it with this run's own numbers
    const int j = a.f_beam[c * k + lane], word = a.f_word[c * k + lane], g = a.f_gate[c * k + lane];
    const int row = c * cur + j;
    float sc;
    if (s_full[j]) {
      const float wl = row_logp(a.logits, a.ld, a.row_max, a.row_lsum, a.forced, row, word);
      sc = __fadd_rn(s_seq[j], __fadd_rn(wl, a.gate_lp[row * 2 + g]));
    } else {
      sc = (word == 0) ? s_seq[j] : -999.f;
    }
    s_pb[lane] = j; s_pw[lane] = word; s_pg[lane] = g; s_ps[lane] = sc;
  }
  __syncwarp();

  if (lane < k && write) {
    const int j = s_pb[lane], word = s_pw[lane], g = s_pg[lane];
    const int row = c * cur + j;
    const int o = c * k + lane;
    // per-token log-probs of the pick, in slot order, masked by the parent's sticky masks (:145,175-177)
    float lw = row_logp(a.logits, a.ld, a.row_max, a.row_lsum, a.forced, row, word);
    float lg = a.gate_lp[row * 2 + g];
    if (a.t > 0) { lw *= s_m0[j]; lg *= s_m1[j]; }
    a.sel_beam[o] = j; a.sel_word[o] = word; a.sel_gate[o] = g;
    a.seq_lp_n[o] = s_ps[lane];
    a.m0n[o] = s_m0[j]; a.m1n[o] = s_m1[j];
    a.hist_parent[o] = j; a.hist_word[o] = word; a.hist_gate[o] = g;
    a.hist_score[o] = s_ps[lane]; a.hist_lpw[o] = lw; a.hist_lpg[o] = lg;
  }
}

// ---------------------------------------------------------------- state advance / reorder
struct AdvanceArgs {
  int rows_new, cur, k;            // new row n' = c*k + i ; parent row = c*cur + parent[n'] (or n' if null)
  const int32_t* parent;
  const int32_t* word32;           // next input token per new row ...
  const int64_t* word64; int64_t word64_stride;   // ... or int64 strided (teacher forcing)
  const int32_t* gate32;           // slot shift per new row, or null
  int fixed_slot;                  // >= 0: set the pointer to this slot (teacher forcing)
  int L, Hp, Ep, V;
  const float *h1n, *c1n, *h2n, *c2n;
  float *h1, *c1, *h2, *c2;
  const int32_t* ptr; int32_t* ptrn;
  int32_t* word_idx;
  // tensor-core twins of h1 / h2 (none on the fp32 path), moved as raw 16-byte vectors: per state up to three arrays
  // (fp16 hi + fp16 lo, or fp16 hi + e4m3 hi8 + e4m3 lo8) of `tw_vec[i]` vectors per row
  int n_tw;
  const uint4* tw_src[8]; uint4* tw_dst[8]; int tw_vec[8];
};

// copy the state of parent row p into new row n, record the next input word, update the slot pointer
__device__ __forceinline__ void advance_row(const AdvanceArgs& a, int n, int p, int64_t w, int gate_shift) {
  const size_t so = (size_t)p * a.Hp, dof = (size_t)n * a.Hp;
  for (int i = threadIdx.x * 4; i < a.Hp; i += blockDim.x * 4) {
    if (a.h1n != nullptr) {        // fp32 h only where somebody reads it (FFMA twin)
      *reinterpret_cast<float4*>(a.h1 + dof + i) = *reinterpret_cast<const float4*>(a.h1n + so + i);
      *reinterpret_cast<float4*>(a.h2 + dof + i) = *reinterpret_cast<const float4*>(a.h2n + so + i);
    }
    *reinterpret_cast<float4*>(a.c1 + dof + i) = *reinterpret_cast<const float4*>(a.c1n + so + i);
    *reinterpret_cast<float4*>(a.c2 + dof + i) = *reinterpret_cast<const float4*>(a.c2n + so + i);
  }
  w = w < 0 ? 0 : (w >= a.V ? a.V - 1 : w);
  for (int q = 0; q < a.n_tw; ++q) {
    const int nv = a.tw_vec[q];
    const uint4* src = a.tw_src[q] + (size_t)p * nv;
    uint4* dst = a.tw_dst[q] + (size_t)n * nv;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) dst[i] = src[i];
  }
  if (threadIdx.x == 0) {
    a.word_idx[n] = (int32_t)w;
    int s;
    if (a.fixed_slot >= 0) s = a.fixed_slot;
    else {
      s = a.ptr[p] + gate_shift;                               // ctrl_det_idxs + prev gate, clamped
      s = s < 0 ? 0 : (s > a.L - 1 ? a.L - 1 : s);             // (controllable_captioning.py:139-140)
    }
    a.ptrn[n] = s;
  }
}

__global__ void __launch_bounds__(256) k_advance(const AdvanceArgs a) {
  const int n = blockIdx.x;
  const int c = n / a.k;
  const int p = a.parent != nullptr ? c * a.cur + a.parent[n] : n;
  const int64_t w = a.word32 != nullptr ? (int64_t)a.word32[n] : a.word64[(size_t)n * a.word64_stride];
  advance_row(a, n, p, w, a.gate32 != nullptr ? a.gate32[n] : 0);
}

// beam selection fused with the reorder of the beam states.  Grid (captions, k): every CTA of a caption
// repeats the (cheap, deterministic) selection with its warp 0 — only CTA y = 0 records it — and then
// moves ONE new beam row, so the copy keeps captions x k CTAs of parallelism without a second launch.
__global__ void __launch_bounds__(256) k_beam_step(const BeamArgs b, const AdvanceArgs a, int do_advance) {
  __shared__ BeamSmem sh;
  const int c = blockIdx.x, i = blockIdx.y;
  pdl_trigger();
  pdl_wait();
  if (threadIdx.x < 32) beam_select_warp(b, sh, c, threadIdx.x, i == 0);
  __syncthreads();
  if (!do_advance) return;
  advance_row(a, c * b.k + i, c * b.cur + sh.pb[i], (int64_t)sh.pw[i], sh.pg[i]);
}

// zero state, slot 0, input word = bos   (init_state, controllable_captioning.py:109-115, :136)
__global__ void k_state_init(float* h1, float* c1, float* h2, float* c2, int32_t* word_idx, int32_t* ptr,
                             int bos, int Hp, TwinOut h1b, TwinOut h2b) {
  const int n = blockIdx.x;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int i = threadIdx.x * 4; i < Hp; i += blockDim.x * 4) {
    const size_t o = (size_t)n * Hp + i;
    *reinterpret_cast<float4*>(h1 + o) = z; *reinterpret_cast<float4*>(c1 + o) = z;
    *reinterpret_cast<float4*>(h2 + o) = z; *reinterpret_cast<float4*>(c2 + o) = z;
    store_twin4(h1b, o, z); store_twin4(h2b, o, z);       // (all-zero bit patterns in fp16 and e4m3 alike)
  }
  if (threadIdx.x == 0) { ptr[n] = 0; word_idx[n] = bos; }
}

__global__ void k_words_from_i64(const int64_t* words, int32_t* word_idx, int rows, int V) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= rows) return;
  int64_t w = words[n];
  w = w < 0 ? 0 : (w >= V ? V - 1 : w);
  word_idx[n] = (int32_t)w;
}

// greedy pick of both heads (CaptioningModel.test, CaptioningModel.py:47): first maximum wins
__global__ void k_greedy_pick(const int32_t* cand, const float* gate_lp, int32_t* sel_word,
                              int32_t* sel_gate, int64_t* out_words, int64_t* out_gates, int rows,
                              int t, int T) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= rows) return;
  const int w = cand[n * VSR_MAX_BEAM];
  const int g = gate_lp[n * 2 + 1] > gate_lp[n * 2 + 0] ? 1 : 0;
  sel_word[n] = w; sel_gate[n] = g;
  out_words[(size_t)n * T + t] = w; out_gates[(size_t)n * T + t] = g;
}

// ---------------------------------------------------------------- multinomial sampling (CaptioningModel.sample_rl)
// Philox4x32-10 counter-based generator: the draw of (seed, caption, step, draw, vocabulary entry) never depends on
// launch shape.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const unsigned hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const unsigned hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u; key.y += 0xBB67AE85u;
  }
  return ctr;
}
__device__ __forceinline__ float u01(unsigned x) { return ((float)(x >> 8) + 0.5f) * (1.f / 16777216.f); }   // (0, 1)

struct SampleArgs {
  const float* logits; int ld, V;
  const float* row_max; const float* row_lsum; const float* gate_lp;
  const int32_t* forced;          // [rows] forced word or -1 (verb forcing), or null
  unsigned long long seed;
  int t, T, n;                    // step, steps, draws per caption (row = caption * n + draw)
  float tau; int top_k; float top_p;
  int32_t *sel_word, *sel_gate;
  int64_t *out_words, *out_gates; float *lp_words, *lp_gates;
};

constexpr int SP_THREADS = 256;
// masses of the top-p select as fixed point (x 2^47): integer sums are exact, so the shared-memory histograms and the
// totals do not depend on the order the atomics land in, and a draw depends on (seed, caption, draw, step, row) alone
constexpr float SP_FIX = 140737488355328.f;   // 2^47; a row of <= 49152 masses <= 1 sums below 2^63

// z = x / tau (x itself at tau = 1), kept finite: at a tiny tau the quotient would overflow to inf and z - max z to NaN
__device__ __forceinline__ float sp_z(float x, float tau) {
  return tau == 1.f ? x : fminf(fmaxf(__fdiv_rn(x, tau), -FLT_MAX), FLT_MAX);
}

// the vocabulary entry of this row whose key is `key`, at 1-based rank r (1 <= r <= number of such entries) among the
// entries of that key in index order.  Tiles of SP_THREADS consecutive entries (conflict-free shared loads), a ballot
// per warp and one barrier per tile; stops at the tile that holds the entry.
__device__ int sp_nth_tie(const float* s_x, int V, unsigned key, unsigned r, unsigned (*s_cnt)[SP_THREADS / 32],
                          int* s_res) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) *s_res = V - 1;
  unsigned base = 0;
  for (int v0 = 0, it = 0; v0 < V; v0 += SP_THREADS, ++it) {
    const int v = v0 + tid;
    const bool hit = v < V && orderable(s_x[v]) == key;
    const unsigned bal = __ballot_sync(0xffffffffu, hit);
    if (lane == 0) s_cnt[it & 1][warp] = __popc(bal);
    __syncthreads();           // (double-buffered counts: the next tile's writes follow this barrier)
    unsigned before_warp = 0, tile = 0;
#pragma unroll
    for (int w = 0; w < SP_THREADS / 32; ++w) {
      const unsigned cw = s_cnt[it & 1][w];
      before_warp += w < warp ? cw : 0u;
      tile += cw;
    }
    if (hit && base + before_warp + __popc(bal & ((1u << lane) - 1u)) + 1u == r) *s_res = v;
    base += tile;
    if (base >= r) break;      // block-uniform
  }
  __syncthreads();
  const int res = *s_res;
  __syncthreads();
  return res;
}

// hist[bin] += val, summed first over the active lanes of the warp that hit the same bin: logits of one row share
// their high key bits, so plain per-lane atomics would serialise on one or two bins.  Integer sums: exact in any order.
template <typename T>
__device__ __forceinline__ void sp_hist_add(T* hist, unsigned bin, T val) {
  namespace cg = cooperative_groups;
  const cg::coalesced_group g = cg::labeled_partition(cg::coalesced_threads(), bin);
  const T sum = cg::reduce(g, val, cg::plus<T>());
  if (g.thread_rank() == 0) atomicAdd(&hist[bin], sum);
}

// Warp 0 walks a 256-bin histogram from the highest digit down and finds the bin in which the running total reaches
// `need` (1 <= need <= total).  Returns the digit; `need` becomes what is still needed inside that bin.
template <typename T>
__device__ __forceinline__ int sp_pick_digit(const T* hist, T& need) {
  const int lane = threadIdx.x & 31;
  T part = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) part += hist[255 - (lane * 8 + i)];
  T incl = part;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const T y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
  const T excl = incl - part;
  const unsigned hit = __ballot_sync(0xffffffffu, excl < need && need <= incl);
  const int src = __ffs(hit) - 1;
  int digit = 0;
  T left = need - excl;
  if (lane == src) {
    for (int i = 0; i < 8; ++i) {
      const T h = hist[255 - (lane * 8 + i)];
      if (left <= h) { digit = 255 - (lane * 8 + i); break; }
      left -= h;
    }
  }
  digit = __shfl_sync(0xffffffffu, digit, src);
  need = __shfl_sync(0xffffffffu, left, src);
  return digit;
}

// Truncated draws: stage row n in s_x and find the (key, index) bound of P.  K (top-k) and P (top-p) are prefixes of
// the order (x desc, index asc), found without sorting: radix selects on orderable(x) in 8-bit digits, 256-bin
// histograms of counts (K) and of exp masses (P), the entries of the boundary value taken in index order.
__device__ void sp_bounds(const SampleArgs& a, int n, const float* x, float* s_x, unsigned& pkey, int& pidx) {
  __shared__ unsigned s_hc[256], s_cnt[2][SP_THREADS / 32];
  __shared__ unsigned long long s_hm[256], s_need;
  __shared__ int s_res;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, V = a.V;
  const float tau = a.tau;
  for (int v = tid * 4; v < V; v += SP_THREADS * 4)
    *reinterpret_cast<float4*>(s_x + v) = *reinterpret_cast<const float4*>(x + v);   // rows are padded to 4 columns
  __syncthreads();
  // ---- K: the first min(top_k, V) entries
  if (a.top_k > 0 && a.top_k < V) {
    unsigned need = (unsigned)a.top_k, prefix = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
      const unsigned hmask = shift == 24 ? 0u : 0xffffffffu << (shift + 8);
      s_hc[tid] = 0u;
      __syncthreads();
      for (int v = tid; v < V; v += SP_THREADS) {
        const unsigned k = orderable(s_x[v]);
        if ((k & hmask) == prefix) sp_hist_add(s_hc, (k >> shift) & 255u, 1u);
      }
      __syncthreads();
      if (warp == 0) {
        const int d = sp_pick_digit(s_hc, need);
        if (lane == 0) { s_cnt[0][0] = prefix | ((unsigned)d << shift); s_cnt[0][1] = need; }
      }
      __syncthreads();
      prefix = s_cnt[0][0]; need = s_cnt[0][1];
      __syncthreads();
    }
    pkey = prefix;
    pidx = sp_nth_tie(s_x, V, prefix, need, s_cnt, &s_res);
  }
  // ---- P: the shortest prefix of K whose mass exp(z - max z) reaches top_p of K's
  if (a.top_p < 1.f) {
    const unsigned kkey = pkey; const int kidx = pidx;
    const float zmax = sp_z(a.row_max[n], tau);
    auto mass = [&](float xv) { return (unsigned long long)__float2ull_rz(expf(sp_z(xv, tau) - zmax) * SP_FIX); };
    unsigned long long need = 0ull;
    unsigned pre = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
      const unsigned hmask = shift == 24 ? 0u : 0xffffffffu << (shift + 8);
      s_hm[tid] = 0ull;
      __syncthreads();
      for (int v = tid; v < V; v += SP_THREADS) {
        const float xv = s_x[v];
        const unsigned k = orderable(xv);
        if ((k & hmask) == pre && (k > kkey || (k == kkey && v <= kidx))) sp_hist_add(s_hm, (k >> shift) & 255u, mass(xv));
      }
      __syncthreads();
      if (warp == 0) {
        if (shift == 24) {     // the first histogram holds all of K: need = ceil(top_p * mass(K)) >= 1 (max z has 2^47)
          unsigned long long tot = 0ull;
#pragma unroll
          for (int i = 0; i < 8; ++i) tot += s_hm[lane * 8 + i];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
          need = (unsigned long long)ceil((double)a.top_p * (double)tot);
        }
        const int d = sp_pick_digit(s_hm, need);
        if (lane == 0) { s_cnt[0][0] = pre | ((unsigned)d << shift); s_need = need; }
      }
      __syncthreads();
      pre = s_cnt[0][0]; need = s_need;
      __syncthreads();
    }
    // every entry of the boundary value has the same mass: take as many of them, in index order, as `need` asks
    const float xb = __uint_as_float((pre & 0x80000000u) ? (pre & 0x7fffffffu) : ~pre);
    const unsigned long long mb = mass(xb);
    pkey = pre;
    pidx = sp_nth_tie(s_x, V, pre, (unsigned)((need + mb - 1) / mb), s_cnt, &s_res);
  }
}

// One CTA per row: word ~ Categorical(softmax(z)), z = logits / tau, restricted to the top-k / top-p set P, by the
// Gumbel-max trick (argmax over P of z + G, G = -log(-log u), draws v with probability exp(z_v) / sum_P exp), gate ~
// Categorical(exp(gate_lp)); log-probs of the draws under the model's untempered distributions, as
// torch.distributions.Categorical(logits=out).log_prob(sample) returns them (CaptioningModel.py:66-70).  A forced row
// (verb forcing, step_v) takes its forced word and gate 1, both with log-prob 0.
// TRUNC = false (no top-k / top-p): the row is read once from global memory (L2: the vocabulary GEMM just wrote it), with
// no shared-memory staging or select state.  TRUNC = true: sp_bounds stages the row in dynamic shared memory and finds
// P; v is in P when orderable(x_v) > key, or == key and v <= index.  Register bounds: 40 for the untruncated pick (6 CTAs
// per SM, as before truncation existed), 64 for the truncated one.
template <bool TRUNC>
__global__ void __launch_bounds__(SP_THREADS, TRUNC ? 4 : 6) k_sample_pick(const SampleArgs a) {
  __shared__ float s_v[SP_THREADS / 32];
  __shared__ int s_i[SP_THREADS / 32];
  const int n = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = n / a.n, j = n - c * a.n, V = a.V;
  const float* x = a.logits + (size_t)n * a.ld;
  const uint2 key = make_uint2((unsigned)a.seed, (unsigned)(a.seed >> 32));
  const size_t o = (size_t)n * a.T + a.t;
  const int forced = a.forced != nullptr ? a.forced[n] : -1;
  if (forced >= 0) {        // step_v: out = 0 at the forced word, gate = [-1e3, 0]
    if (tid == 0) {
      a.sel_word[n] = forced; a.sel_gate[n] = 1;
      a.out_words[o] = forced; a.out_gates[o] = 1; a.lp_words[o] = 0.f; a.lp_gates[o] = 0.f;
    }
    return;
  }
  const float tau = a.tau;
  const float* src = x;
  unsigned pk = 0u; int pi = 0x7fffffff;           // bound of P
  if constexpr (TRUNC) {
    extern __shared__ __align__(16) float s_x[];
    sp_bounds(a, n, x, s_x, pk, pi);
    src = s_x;
  }
  // ---- draw: Gumbel-max over P, lanes of one Philox block = 4 consecutive vocabulary entries
  float bv = -INFINITY; int bi = 0x7fffffff;
  for (int v0 = tid * 4; v0 < V; v0 += SP_THREADS * 4) {
    const float4 q = *reinterpret_cast<const float4*>(src + v0);
    const float xs[4] = {q.x, q.y, q.z, q.w};
    bool in[4];
    bool any = false;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const unsigned k = orderable(xs[e]);
      in[e] = v0 + e < V && (!TRUNC || k > pk || (k == pk && v0 + e <= pi));
      any |= in[e];
    }
    if (!any) continue;
    const uint4 r = philox4x32_10(make_uint4((unsigned)(v0 >> 2), (unsigned)c, (unsigned)a.t, 2u * (unsigned)j), key);
    const unsigned rs[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (!in[e]) continue;
      const float g = -logf(-logf(u01(rs[e])));
      const float sc = sp_z(xs[e], tau) + g;
      if (sc > bv) { bv = sc; bi = v0 + e; }
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
    if (before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
  }
  if (lane == 0) { s_v[warp] = bv; s_i[warp] = bi; }
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < SP_THREADS / 32; ++w) if (before(s_v[w], s_i[w], bv, bi)) { bv = s_v[w]; bi = s_i[w]; }
    const int word = bi < V ? bi : V - 1;
    const float lw = (x[word] - a.row_max[n]) - a.row_lsum[n];
    // gate: two categories with log-probs gate_lp[n]; counter word 2j + 1 keeps this draw apart from the vocabulary's
    const uint4 r = philox4x32_10(make_uint4(0u, (unsigned)c, (unsigned)a.t, 2u * (unsigned)j + 1u), key);
    const float g0 = a.gate_lp[(size_t)n * 2], g1 = a.gate_lp[(size_t)n * 2 + 1];
    const int gate = u01(r.x) < expf(g0) ? 0 : 1;
    a.sel_word[n] = word; a.sel_gate[n] = gate;
    a.out_words[o] = word; a.out_gates[o] = gate;
    a.lp_words[o] = lw; a.lp_gates[o] = gate == 0 ? g0 : g1;
  }
}

// final ordering of the beams by accumulated score (stable, descending) and unroll of the
// back-pointers (CaptioningModel.py:182-194 / 279-293).  One CTA per caption: the caption's [T][k] history is
// staged in shared memory with coalesced loads, so the serial pointer chase never waits on global memory.
// path_row (optional, [b][out_size][T]): the step-t row whose distributions produced token t of the returned beam.
__global__ void __launch_bounds__(64) k_backtrack(int b, int k, int T, int out_size, const float* seq_lp,
                                                  const int32_t* hist_parent, const int32_t* hist_word,
                                                  const int32_t* hist_gate, const float* hist_lpw, const float* hist_lpg,
                                                  int64_t* out_words, int64_t* out_gates, float* lp_words, float* lp_gates,
                                                  int32_t* path_row) {
  extern __shared__ __align__(16) unsigned char bt_smem[];      // 5 arrays of T*k 4-byte entries (<= 40 KB)
  int32_t* s_par = reinterpret_cast<int32_t*>(bt_smem);
  int32_t* s_wrd = s_par + T * k;
  int32_t* s_gat = s_wrd + T * k;
  float* s_lpw = reinterpret_cast<float*>(s_gat + T * k);
  float* s_lpg = s_lpw + T * k;
  __shared__ float s_seq[VSR_MAX_BEAM];
  const int c = blockIdx.x;
  for (int i = threadIdx.x; i < T * k; i += blockDim.x) {
    const int t = i / k, j = i - t * k;
    const size_t hi = ((size_t)t * b + c) * k + j;
    s_par[i] = hist_parent[hi]; s_wrd[i] = hist_word[hi]; s_gat[i] = hist_gate[hi];
    s_lpw[i] = hist_lpw[hi]; s_lpg[i] = hist_lpg[hi];
  }
  if (threadIdx.x < k) s_seq[threadIdx.x] = seq_lp[c * k + threadIdx.x];
  __syncthreads();
  const int o = threadIdx.x;
  if (o >= out_size) return;
  int order[VSR_MAX_BEAM];
  for (int i = 0; i < k; ++i) order[i] = i;
  for (int i = 1; i < k; ++i) {   // insertion sort, stable, descending
    const int oi = order[i];
    const float v = s_seq[oi];
    int j = i - 1;
    while (j >= 0 && s_seq[order[j]] < v) { order[j + 1] = order[j]; --j; }
    order[j + 1] = oi;
  }
  const int final_slot = order[o];
  int slot = final_slot;
  const size_t ob = ((size_t)c * out_size + o) * T;
  for (int t = T - 1; t >= 0; --t) {
    out_words[ob + t] = s_wrd[t * k + slot];
    out_gates[ob + t] = s_gat[t * k + slot];
    // log-probs are NOT back-tracked: slot order at step t, permuted by the final sort only
    lp_words[ob + t] = s_lpw[t * k + final_slot];
    lp_gates[ob + t] = s_lpg[t * k + final_slot];
    slot = s_par[t * k + slot];
    // the attention, unlike the log-probs, follows the back-pointers: rows of step t are c * cur_t + parent slot
    if (path_row != nullptr) path_row[ob + t] = c * (t == 0 ? 1 : k) + slot;
  }
}

// attention of the returned sequences from the per-step capture: out row i (caption * out_size + beam) at step t reads
// captured row path_row[i][t] of step t, or row i itself when path_row is null (one row per caption: greedy, sampling,
// teacher forcing).  One warp per (i, t).
__global__ void __launch_bounds__(128) k_attn_gather(const float* __restrict__ alpha_ws, const int32_t* __restrict__ slot_ws,
                                                     int64_t step_rows, const int32_t* __restrict__ path_row, int n_out, int T,
                                                     int W, float* __restrict__ alpha, int32_t* __restrict__ slot) {
  const int lane = threadIdx.x & 31;
  const int item = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (item >= n_out * T) return;
  const int i = item / T, t = item - i * T;
  const int64_t row = path_row != nullptr ? path_row[item] : i;
  const int64_t src = (int64_t)t * step_rows + row;
  for (int j = lane; j < W; j += 32) alpha[(size_t)item * W + j] = alpha_ws[(size_t)src * W + j];
  if (lane == 0) slot[item] = slot_ws[src];
}

}  // namespace

static TwinOut pp(const Ctx* c, const F16Pair& b) { return twin_out(&b, c->use_tc); }

int launch_state_init(Ctx* c, int rows, cudaStream_t st) {
  k_state_init<<<rows, 256, 0, st>>>(c->h1, c->c1, c->h2, c->c2, c->word_idx, c->ptr, c->d.bos_idx, c->Hp,
                                     pp(c, c->h1_b), pp(c, c->h2_b));
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

int launch_words(Ctx* c, const int64_t* words, int rows, cudaStream_t st) {
  k_words_from_i64<<<(rows + 127) / 128, 128, 0, st>>>(words, c->word_idx, rows, c->V);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

static void fill_advance(Ctx* c, AdvanceArgs& a) {
  a.L = c->L; a.Hp = c->Hp; a.Ep = c->Ep; a.V = c->V;
  a.h1n = c->state_h32 ? c->h1n : nullptr; a.c1n = c->c1n; a.h2n = c->state_h32 ? c->h2n : nullptr; a.c2n = c->c2n;
  a.h1 = c->h1; a.c1 = c->c1; a.h2 = c->h2; a.c2 = c->c2;
  a.ptr = c->ptr; a.ptrn = c->ptrn; a.word_idx = c->word_idx;
  a.n_tw = 0;
  if (c->use_tc) {
    auto add = [&](const void* src, void* dst, int bytes_per_elem) {
      if (src == nullptr || dst == nullptr) return;
      a.tw_src[a.n_tw] = (const uint4*)src; a.tw_dst[a.n_tw] = (uint4*)dst; a.tw_vec[a.n_tw] = c->Hp * bytes_per_elem / 16;
      ++a.n_tw;
    };
    const F16Pair* src[2] = {&c->h1n_b, &c->h2n_b};
    F16Pair* dst[2] = {&c->h1_b, &c->h2_b};
    for (int q = 0; q < 2; ++q) {
      add(src[q]->hi, dst[q]->hi, 2); add(src[q]->lo, dst[q]->lo, 2);
      add(src[q]->hi8, dst[q]->hi8, 1); add(src[q]->lo8, dst[q]->lo8, 1);
    }
  }
}

// beam selection of step t and (unless it is the last step) the state reorder for step t+1, one launch
int launch_beam_step(Ctx* c, int t, int b, int cur, int k, int64_t eos0, int64_t eos1, const int32_t* f_beam,
                     const int32_t* f_word, const int32_t* f_gate, bool advance, cudaStream_t st) {
  PhaseScope ps(c, PH_BEAM, st);
  BeamArgs a{};
  a.t = t; a.b = b; a.cur = cur; a.k = k; a.V = c->V; a.eos0 = eos0; a.eos1 = eos1;
  a.logits = c->logits; a.ld = c->NE; a.row_max = c->row_max; a.row_lsum = c->row_lsum;
  a.forced = c->forced; a.cand = c->cand; a.gate_lp = c->gate_lp;
  a.seq_lp = c->seq_lp; a.seq_lp_n = c->seq_lp_n;
  a.m0 = c->m0; a.m1 = c->m1; a.m0n = c->m0n; a.m1n = c->m1n;
  a.prev_word = c->sel_word; a.prev_gate = c->sel_gate;
  a.sel_beam = c->sel_beam_n; a.sel_word = c->sel_word_n; a.sel_gate = c->sel_gate_n;
  const size_t off = (size_t)t * b * k;
  a.hist_parent = c->hist_parent + off; a.hist_word = c->hist_word + off; a.hist_gate = c->hist_gate + off;
  a.hist_score = c->hist_score + off; a.hist_lpw = c->hist_lpw + off; a.hist_lpg = c->hist_lpg + off;
  a.f_beam = f_beam; a.f_word = f_word; a.f_gate = f_gate;
  AdvanceArgs ad{};
  ad.rows_new = b * k; ad.cur = cur; ad.k = k; ad.fixed_slot = -1;
  fill_advance(c, ad);
  VSR_CHECK_CUDA(launch_k(k_beam_step, dim3(b, advance ? k : 1), dim3(256), 0, st, c->use_pdl && (c->pdl_mode & 2), a, ad, advance ? 1 : 0));
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  std::swap(c->sel_beam, c->sel_beam_n);
  std::swap(c->sel_word, c->sel_word_n);
  std::swap(c->sel_gate, c->sel_gate_n);
  std::swap(c->seq_lp, c->seq_lp_n);
  std::swap(c->m0, c->m0n);
  std::swap(c->m1, c->m1n);
  if (advance) std::swap(c->ptr, c->ptrn);
  return VSR_OK;
}

static int launch_advance(Ctx* c, AdvanceArgs& a, cudaStream_t st) {
  fill_advance(c, a);
  k_advance<<<a.rows_new, 256, 0, st>>>(a);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  std::swap(c->ptr, c->ptrn);
  return VSR_OK;
}

int launch_commit_identity(Ctx* c, int rows, const int64_t* next_words, int64_t word_stride,
                           int next_slot, cudaStream_t st) {
  PhaseScope ps(c, PH_REORDER, st);
  AdvanceArgs a{};
  a.rows_new = rows; a.cur = 1; a.k = 1;
  a.parent = nullptr;
  if (next_words != nullptr) { a.word64 = next_words; a.word64_stride = word_stride; a.gate32 = nullptr; }
  else { a.word32 = c->sel_word; a.gate32 = c->sel_gate; }
  a.fixed_slot = next_slot;
  return launch_advance(c, a, st);
}

int launch_greedy_pick(Ctx* c, int rows, int t, int T, int64_t* out_words, int64_t* out_gates,
                       cudaStream_t st) {
  PhaseScope ps(c, PH_BEAM, st);
  k_greedy_pick<<<(rows + 127) / 128, 128, 0, st>>>(c->cand, c->gate_lp, c->sel_word, c->sel_gate,
                                                    out_words, out_gates, rows, t, T);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

int launch_sample_pick(Ctx* c, int rows, int t, int T, const VsrSampleParams& p, int64_t* out_words,
                       int64_t* out_gates, float* lp_words, float* lp_gates, cudaStream_t st) {
  PhaseScope ps(c, PH_BEAM, st);
  SampleArgs a{};
  a.logits = c->logits; a.ld = c->NE; a.V = c->V;
  a.row_max = c->row_max; a.row_lsum = c->row_lsum; a.gate_lp = c->gate_lp;
  a.forced = p.use_verbs ? c->forced : nullptr;
  a.seed = (unsigned long long)p.seed; a.t = t; a.T = T; a.n = p.n;
  a.tau = p.temperature; a.top_k = p.top_k; a.top_p = p.top_p;
  const bool trunc = (p.top_k > 0 && p.top_k < c->V) || p.top_p < 1.f;
  a.sel_word = c->sel_word; a.sel_gate = c->sel_gate;
  a.out_words = out_words; a.out_gates = out_gates; a.lp_words = lp_words; a.lp_gates = lp_gates;
  if (!trunc) {
    k_sample_pick<false><<<rows, SP_THREADS, 0, st>>>(a);
  } else {
    if (!c->sample_attr_set) {     // up to 192 KB at the largest vocabulary (per device, hence per handle)
      VSR_CHECK_CUDA(cudaFuncSetAttribute(k_sample_pick<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * 1024 * 4));
      c->sample_attr_set = true;
    }
    k_sample_pick<true><<<rows, SP_THREADS, sizeof(float) * (size_t)round_up(c->V, 4), st>>>(a);
  }
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

int launch_backtrack(Ctx* c, int b, int k, int T, int out_size, int64_t* out_words,
                     int64_t* out_gates, float* lp_words, float* lp_gates, int32_t* path_row, cudaStream_t st) {
  PhaseScope ps(c, PH_FINAL, st);
  VSR_REQUIRE(T <= VSR_MAX_SEQ_LEN, VSR_EINVAL, "seq_len=%d > %d unsupported by the back-track kernel", T, VSR_MAX_SEQ_LEN);
  // final scores come from the history slice of the last step, NOT from the ping-pong buffer c->seq_lp: a replayed
  // CUDA graph bakes in the ping-pong parity of its capture, which need not be the host's current one (odd seq_len)
  k_backtrack<<<b, 64, (size_t)T * k * 20, st>>>(b, k, T, out_size, c->hist_score + (size_t)(T - 1) * b * k, c->hist_parent, c->hist_word,
                                            c->hist_gate, c->hist_lpw, c->hist_lpg, out_words, out_gates,
                                            lp_words, lp_gates, path_row);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

int launch_attn_gather(Ctx* c, const int32_t* path_row, int n_out, int T, float* alpha, int32_t* slot, cudaStream_t st) {
  const int items = n_out * T;
  k_attn_gather<<<(items + 3) / 4, 128, 0, st>>>(c->attn_alpha, c->attn_slot, c->attn_step_rows, path_row, n_out, T,
                                                 c->attn_R + 1, alpha, slot);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

}  // namespace vsr
