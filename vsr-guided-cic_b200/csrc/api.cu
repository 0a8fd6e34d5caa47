// C-ABI entry points of libvsrdec (include/vsrdec.h): context life-cycle, workspace
// management and the decode drivers (beam search, teacher-forced forward, greedy, single step).
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace vsr {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int dev_alloc(Ctx* c, void** p, size_t bytes, bool zero) {
  *p = nullptr;
  if (bytes == 0) bytes = 16;
  cudaError_t e = cudaMalloc(p, bytes);
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    cudaGetLastError();
    return VSR_ENOMEM;
  }
  c->owned.push_back(*p);
  c->epoch++;
  if (zero) VSR_CHECK_CUDA(cudaMemset(*p, 0, bytes));
  return VSR_OK;
}

static void dev_free(Ctx* c, void* p) {
  if (p == nullptr) return;
  auto it = std::find(c->owned.begin(), c->owned.end(), p);
  if (it != c->owned.end()) c->owned.erase(it);
  c->epoch++;
  cudaFree(p);
}

PhaseScope::PhaseScope(Ctx* c_, int id_, cudaStream_t st_) : c(c_), id(id_), st(st_) {
  c->phases[id].launches++;
  if (!c->profiling) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); c->phases[id].ev.push_back(e); }
}
PhaseScope::~PhaseScope() {
  if (!c->profiling) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); c->phases[id].ev.push_back(e); }
}

static const char* kPhaseNames[PH_COUNT] = {
    "prologue", "gemm_a_lstm1_gates", "lstm1_pointwise", "gemm_b_sentinel_h1proj", "gate_pointwise",
    "gemm_c_att_ga", "attend_gate", "gemm_d_lstm2_gates", "lstm2_pointwise", "gemm_e_vocab",
    "softmax_topk", "beam_select", "state_reorder", "backtrack"};

static void reset_phases(Ctx* c) {
  for (int i = 0; i < PH_COUNT; ++i) {
    for (cudaEvent_t e : c->phases[i].ev) cudaEventDestroy(e);
    c->phases[i].ev.clear();
    c->phases[i].launches = 0;
  }
}

#define ALLOC_F(ptr, count) VSR_TRY(dev_alloc(c, (void**)&(ptr), sizeof(float) * (size_t)(count)))

// (re)allocate a fp16 hi/lo twin of a [rows][ld] fp32 matrix and build its TMA tensor maps
// padded row count of a weight whose GEMM may run with N tile `bn` or `alt_bn`
static int pad_rows(int n_valid, int bn, int alt_bn) {
  int r = round_up(n_valid, bn);
  if (alt_bn > 0) r = std::max(r, round_up(n_valid, alt_bn));
  return round_up(r, 128);
}

// kind of twin set: fp16 hi + fp16 residual (f16x3 GEMMs) or fp16 hi + e4m3 hi8 / lo8 (f16+f8x2 GEMMs)
enum PairKind { PAIR_F16X3 = 0, PAIR_F8 = 1 };
static PairKind step_kind(const Ctx* c) { return c->gemm_f8 ? PAIR_F8 : PAIR_F16X3; }

int alloc_pair(Ctx* c, F16Pair* b, int rows, int ld, int box_rows, PairKind kind, bool weight = false, int n_valid = 0,
               int alt_bn = 0) {
  dev_free(c, b->hi); dev_free(c, b->lo); dev_free(c, b->hi8); dev_free(c, b->lo8);
  b->hi = b->lo = b->hi8 = b->lo8 = nullptr;
  if (!c->use_tc) return VSR_OK;
  VSR_TRY(dev_alloc(c, &b->hi, (size_t)rows * ld * 2));
  b->rows = rows; b->ld = ld; b->box_rows = box_rows;
  VSR_TRY(make_tmap_f16(b->map_hi, b->hi, rows, ld, ld, box_rows));
  if (kind == PAIR_F16X3) {
    VSR_TRY(dev_alloc(c, &b->lo, (size_t)rows * ld * 2));
    VSR_TRY(make_tmap_f16(b->map_lo, b->lo, rows, ld, ld, box_rows));
  } else {
    VSR_TRY(dev_alloc(c, &b->hi8, (size_t)rows * ld));
    VSR_TRY(dev_alloc(c, &b->lo8, (size_t)rows * ld));
    VSR_TRY(make_tmap_u8(b->map8_hi, b->hi8, rows, ld, ld, box_rows));
    VSR_TRY(make_tmap_u8(b->map8_lo, b->lo8, rows, ld, ld, box_rows));
  }
  b->act_scale = (!weight && kind == PAIR_F8) ? ACT_SCALE_F8 : 1.f;
  b->n_valid = n_valid > 0 ? n_valid : rows;
  b->alt_bn = alt_bn;
  if (alt_bn > 0) {
    VSR_TRY(make_tmap_f16(b->alt_hi, b->hi, rows, ld, ld, alt_bn));
    if (kind == PAIR_F16X3) {
      VSR_TRY(make_tmap_f16(b->alt_lo, b->lo, rows, ld, ld, alt_bn));
    } else {
      VSR_TRY(make_tmap_u8(b->alt8_hi, b->hi8, rows, ld, ld, alt_bn));
      VSR_TRY(make_tmap_u8(b->alt8_lo, b->lo8, rows, ld, ld, alt_bn));
    }
  }
  if (weight && b->scale == nullptr) VSR_TRY(dev_alloc(c, (void**)&b->scale, 2 * sizeof(float)));
  return VSR_OK;
}

int ensure_rows(Ctx* c, int rows) {
  if (rows <= c->cap_rows) return VSR_OK;
  const int cap = round_up(rows, MPAD);
  float** bufs[] = {&c->h1, &c->c1, &c->h2, &c->c2, &c->h1n, &c->c1n, &c->h2n, &c->c2n, &c->pre1,
                    &c->s_t, &c->g_t, &c->gq, &c->sent, &c->hb, &c->ga, &c->att, &c->pre2, &c->logits, &c->gate_lp,
                    &c->row_max, &c->row_lsum, &c->shift, &c->vpart};
  for (float** p : bufs) { dev_free(c, *p); *p = nullptr; }
  dev_free(c, c->word_idx);
  dev_free(c, c->ptr); dev_free(c, c->ptrn); dev_free(c, c->forced); dev_free(c, c->cand); dev_free(c, c->word_in);
  c->cap_rows = 0;
  const size_t n = cap;
  ALLOC_F(c->h1, n * c->Hp); ALLOC_F(c->c1, n * c->Hp); ALLOC_F(c->h2, n * c->Hp); ALLOC_F(c->c2, n * c->Hp);
  ALLOC_F(c->h1n, n * c->Hp); ALLOC_F(c->c1n, n * c->Hp); ALLOC_F(c->h2n, n * c->Hp); ALLOC_F(c->c2n, n * c->Hp);
  VSR_TRY(dev_alloc(c, (void**)&c->word_idx, sizeof(int32_t) * n));
  ALLOC_F(c->pre1, n * c->NA);
  ALLOC_F(c->s_t, n * c->Hp); ALLOC_F(c->g_t, n * c->Hp); ALLOC_F(c->gq, n * c->Hp);
  ALLOC_F(c->sent, n * c->NB1); ALLOC_F(c->hb, n * c->NB2); ALLOC_F(c->ga, n * c->NC);
  ALLOC_F(c->att, n * c->Fp); ALLOC_F(c->pre2, n * c->ND); ALLOC_F(c->logits, n * c->NE);
  ALLOC_F(c->gate_lp, n * 2); ALLOC_F(c->row_max, n); ALLOC_F(c->row_lsum, n); ALLOC_F(c->shift, n);
  ALLOC_F(c->vpart, n * (size_t)(c->NE / 16) * 2);
  VSR_TRY(dev_alloc(c, (void**)&c->ptr, sizeof(int32_t) * n));
  VSR_TRY(dev_alloc(c, (void**)&c->ptrn, sizeof(int32_t) * n));
  VSR_TRY(dev_alloc(c, (void**)&c->forced, sizeof(int32_t) * n));
  VSR_TRY(dev_alloc(c, (void**)&c->cand, sizeof(int32_t) * n * VSR_MAX_BEAM));
  VSR_TRY(dev_alloc(c, (void**)&c->word_in, sizeof(int64_t) * n));
  const PairKind sk = step_kind(c);
  VSR_TRY(alloc_pair(c, &c->h1_b, cap, c->Hp, MPAD, sk)); VSR_TRY(alloc_pair(c, &c->h2_b, cap, c->Hp, MPAD, sk));
  VSR_TRY(alloc_pair(c, &c->s_t_b, cap, c->Hp, MPAD, sk));
  VSR_TRY(alloc_pair(c, &c->h1n_b, cap, c->Hp, MPAD, sk)); VSR_TRY(alloc_pair(c, &c->g_t_b, cap, c->Hp, MPAD, sk));
  VSR_TRY(alloc_pair(c, &c->att_b, cap, c->Fp, MPAD, sk)); VSR_TRY(alloc_pair(c, &c->h2n_b, cap, c->Hp, MPAD, sk));
  c->cap_rows = cap;
  return VSR_OK;
}

// per-row selection buffers (beam search: caps * VSR_MAX_BEAM slots; greedy and sampling: one per decoded row)
int ensure_sel(Ctx* c, int rows) {
  if (rows <= c->cap_sel) return VSR_OK;
  int32_t** ib[] = {&c->sel_beam, &c->sel_word, &c->sel_gate, &c->sel_beam_n, &c->sel_word_n, &c->sel_gate_n};
  for (int32_t** p : ib) { dev_free(c, *p); *p = nullptr; }
  c->cap_sel = 0;
  for (int32_t** p : ib) VSR_TRY(dev_alloc(c, (void**)p, sizeof(int32_t) * (size_t)rows));
  c->cap_sel = rows;
  return VSR_OK;
}

int ensure_beam_ws(Ctx* c, int caps, int T) {
  VSR_TRY(ensure_sel(c, caps * VSR_MAX_BEAM));
  if (caps <= c->cap_caps && T <= c->cap_T) return VSR_OK;
  caps = std::max(caps, c->cap_caps); T = std::max(T, c->cap_T);
  float** fb[] = {&c->seq_lp, &c->seq_lp_n, &c->m0, &c->m1, &c->m0n, &c->m1n, &c->hist_score, &c->hist_lpw, &c->hist_lpg};
  int32_t** ib[] = {&c->hist_parent, &c->hist_word, &c->hist_gate};
  for (float** p : fb) { dev_free(c, *p); *p = nullptr; }
  for (int32_t** p : ib) { dev_free(c, *p); *p = nullptr; }
  c->cap_caps = 0; c->cap_T = 0;
  const size_t s = (size_t)caps * VSR_MAX_BEAM, hs = s * T;
  ALLOC_F(c->seq_lp, s); ALLOC_F(c->seq_lp_n, s); ALLOC_F(c->m0, s); ALLOC_F(c->m1, s); ALLOC_F(c->m0n, s); ALLOC_F(c->m1n, s);
  ALLOC_F(c->hist_score, hs); ALLOC_F(c->hist_lpw, hs); ALLOC_F(c->hist_lpg, hs);
  VSR_TRY(dev_alloc(c, (void**)&c->hist_parent, sizeof(int32_t) * hs));
  VSR_TRY(dev_alloc(c, (void**)&c->hist_word, sizeof(int32_t) * hs));
  VSR_TRY(dev_alloc(c, (void**)&c->hist_gate, sizeof(int32_t) * hs));
  c->cap_caps = caps; c->cap_T = T;
  return VSR_OK;
}

// n-gram blocking histories of `rows` rows (grow-only; both buffers of the pair)
int ensure_whist(Ctx* c, int rows) {
  if (rows <= c->cap_whist) return VSR_OK;
  dev_free(c, c->whist); dev_free(c, c->whist_n);
  c->whist = c->whist_n = nullptr; c->cap_whist = 0;
  const size_t n = (size_t)rows * c->d.seq_len;
  VSR_TRY(dev_alloc(c, (void**)&c->whist, sizeof(int32_t) * n));
  VSR_TRY(dev_alloc(c, (void**)&c->whist_n, sizeof(int32_t) * n));
  c->cap_whist = rows;
  return VSR_OK;
}

// grow-only capture buffers for a decode of T steps with up to step_rows rows per step (and a back-tracked path of
// path entries); clears what the previous decode left.  Nothing is allocated while capture is off.
static int attn_begin(Ctx* c, int64_t step_rows, int T, size_t path) {
  c->attn_ready = false;
  if (!c->attn_capture) return VSR_OK;
  const size_t n_slot = (size_t)step_rows * T, n_alpha = n_slot * (c->R + 1);
  if (n_alpha > c->cap_attn_alpha) {
    dev_free(c, c->attn_alpha); c->attn_alpha = nullptr; c->cap_attn_alpha = 0;
    ALLOC_F(c->attn_alpha, n_alpha);
    c->cap_attn_alpha = n_alpha;
  }
  if (n_slot > c->cap_attn_slot) {
    dev_free(c, c->attn_slot); c->attn_slot = nullptr; c->cap_attn_slot = 0;
    VSR_TRY(dev_alloc(c, (void**)&c->attn_slot, sizeof(int32_t) * n_slot));
    c->cap_attn_slot = n_slot;
  }
  if (path > c->cap_attn_path) {
    dev_free(c, c->attn_path); c->attn_path = nullptr; c->cap_attn_path = 0;
    VSR_TRY(dev_alloc(c, (void**)&c->attn_path, sizeof(int32_t) * path));
    c->cap_attn_path = path;
  }
  return VSR_OK;
}

// capture outputs of step t: rows of step t start at t * step_rows (null pointers when capture is off)
static void attn_step_io(const Ctx* c, StepIO& io, int t, int64_t step_rows) {
  if (!c->attn_capture) return;
  io.attn_alpha = c->attn_alpha + (size_t)t * step_rows * (c->R + 1);
  io.attn_slot = c->attn_slot + (size_t)t * step_rows;
}

// after a successful decode: what vsr_get_attention returns (n_out rows per step, back-tracked when beam)
static void attn_done(Ctx* c, bool beam, int T, int n_out, int64_t step_rows) {
  c->attn_ready = c->attn_capture;
  c->attn_beam = beam; c->attn_T = T; c->attn_R = c->R; c->attn_n_out = n_out; c->attn_step_rows = step_rows;
}

static int create_impl(const VsrDims* d, const float* const* w, Ctx** out) {
  VSR_REQUIRE(d != nullptr && w != nullptr && out != nullptr, VSR_EINVAL, "vsr_create: null argument");
  VSR_REQUIRE(d->vocab_size > 0 && d->rnn_size > 0 && d->att_size > 0 && d->input_encoding_size > 0 &&
                  d->det_feat_size > 0 && d->seq_len > 0,
              VSR_EINVAL, "vsr_create: non-positive dimension");
  VSR_REQUIRE(d->det_feat_size % 4 == 0 && d->att_size % 4 == 0, VSR_EINVAL,
              "vsr_create: det_feat_size=%d and att_size=%d must be multiples of 4 (128-bit loads)",
              d->det_feat_size, d->att_size);
  VSR_REQUIRE(d->bos_idx >= 0 && d->bos_idx < d->vocab_size, VSR_EINVAL, "vsr_create: bos_idx out of range");
  VSR_REQUIRE(d->vocab_size <= 1024 * 48, VSR_EINVAL,
              "vsr_create: vocab_size=%d > 49152 unsupported (register-resident softmax/top-k row)", d->vocab_size);
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  VSR_REQUIRE(e == cudaSuccess && ndev > 0, VSR_ECUDA,
              "vsr_create: no CUDA device available (%s); libvsrdec has no CPU fallback",
              cudaGetErrorString(e));
  Ctx* c = new Ctx();
  c->d = *d;
  VSR_CHECK_CUDA(cudaGetDevice(&c->device));
  c->V = d->vocab_size; c->E = d->input_encoding_size; c->H = d->rnn_size; c->F = d->det_feat_size; c->A = d->att_size;
  c->Hp = round_up(c->H, KPAD); c->Ep = round_up(c->E, KPAD); c->Fp = round_up(c->F, KPAD); c->Ap = round_up(c->A, KPAD);
  c->NA = 6 * c->Hp;                       // gate-interleaved: 6 gates x Hp units (multiple of 192 and 128)
  // N tiles: 128 by default; the vocabulary projection also gets an alternative tile (144) that the launcher
  // picks when it covers the problem in fewer waves of 148 CTAs (V = 10000 at 500 rows: 280 tiles = 2 waves
  // instead of 316 = 3).  Tiles wider than 192 measured slow on B200 (operand delivery per SM drops), so the
  // h1'/s_t projections stay at 128.
  c->oB1_sa = c->Fp;
  c->NB1v = c->oB1_sa + c->A;
  c->NB1 = pad_rows(c->NB1v, 128, 0);
  c->oB2_ha = c->Hp;
  c->oB2_p2 = c->oB2_ha + c->Ap;
  c->NB2v = c->oB2_p2;                     // (h1' -> LSTM2 gates lives in GEMM-D as a third K segment)
  c->NB2 = pad_rows(c->NB2v, 128, 0);
  c->NC = round_up(c->A, NPAD);
  c->ND = 4 * c->Hp;                       // gate-interleaved: 4 gates x Hp units (multiple of 256)
  c->NE = round_up(c->V, 1152);            // whole tiles for every N tile of the vocabulary GEMM: 128, 144, 192 (lcm 1152)
  c->NVA = round_up(c->A, NPAD);
  c->KA = (d->h2_first_lstm ? c->Hp : 0) + c->Hp;
  c->KD = c->Fp + 2 * c->Hp;
  for (int i = 0; i < PH_COUNT; ++i) c->phases[i].name = kPhaseNames[i];
  *out = c;   // from here on vsr_destroy can clean up a half-built context
  ALLOC_F(c->WA, (size_t)c->NA * c->KA); ALLOC_F(c->WU, (size_t)c->NA * c->Fp); ALLOC_F(c->bU, c->NA);
  ALLOC_F(c->WB1, (size_t)c->NB1 * c->Hp); ALLOC_F(c->bB1, c->NB1);
  ALLOC_F(c->WB2, (size_t)c->NB2 * c->Hp);
  ALLOC_F(c->WC, (size_t)c->NC * c->Hp);
  ALLOC_F(c->WD, (size_t)c->ND * c->KD); ALLOC_F(c->bD, c->ND);
  if (d->img_second_lstm) ALLOC_F(c->WU2, (size_t)c->ND * c->Fp);
  ALLOC_F(c->WE, (size_t)c->NE * c->Hp); ALLOC_F(c->bE, c->NE);
  ALLOC_F(c->Wva, (size_t)c->NVA * c->Fp);
  ALLOC_F(c->v_a, c->Ap); ALLOC_F(c->v_s, c->Ap); ALLOC_F(c->v_g, c->Ap);
  ALLOC_F(c->embed, (size_t)c->V * c->Ep);
  ALLOC_F(c->WAx, (size_t)c->NA * c->Ep); ALLOC_F(c->X, (size_t)c->V * c->NA);
  {
    // VSRDEC_GEMM: "simt" = fp32 FFMA twin for A/B verification of the tcgen05 path; "f16x3" = all three passes of the
    // step GEMMs in fp16 (default: the two residual passes on the fp8 tensor path, "f16+f8x2")
    const char* mode = getenv("VSRDEC_GEMM");
    c->use_tc = !(mode != nullptr && strcmp(mode, "simt") == 0);
    c->gemm_f8 = !(mode != nullptr && strcmp(mode, "f16x3") == 0);
  }
  if (const char* e = getenv("VSRDEC_GRAPH")) c->use_graphs = atoi(e) != 0;
  if (const char* e = getenv("VSRDEC_PDL")) c->use_pdl = atoi(e) != 0;
  // UMMA N tile of the single-CTA kernel: 128 (wider tiles measured slower on B200 for every per-step shape: fewer CTAs
  // in flight, shallower ring).  GEMM-A / GEMM-D tiles are fixed by their fused LSTM epilogues: 6 gates x 32 units = 192,
  // 4 x 32 = 128.  Weight pairs are power-of-two scaled per tensor (F16Pair::scale).
  const PairKind sk = step_kind(c);
  VSR_TRY(alloc_pair(c, &c->WA_b, c->NA, c->KA, 192, sk, true)); VSR_TRY(alloc_pair(c, &c->WB1_b, c->NB1, c->Hp, 128, sk, true, c->NB1v));
  VSR_TRY(alloc_pair(c, &c->WB2_b, c->NB2, c->Hp, 128, sk, true, c->NB2v)); VSR_TRY(alloc_pair(c, &c->WC_b, c->NC, c->Hp, 128, sk, true));
  VSR_TRY(alloc_pair(c, &c->WD_b, c->ND, c->KD, 128, sk, true)); VSR_TRY(alloc_pair(c, &c->WE_b, c->NE, c->Hp, 128, sk, true, c->V, 144));
  if (c->use_tc) {     // CTA-pair kernel for the large-batch launches: 256 x 192 tiles for A and E, 256 x 256 for B, D + C
    VSR_TRY(make_pair_maps(&c->WA_b, 96)); VSR_TRY(make_pair_maps(&c->WB1_b, 128)); VSR_TRY(make_pair_maps(&c->WB2_b, 128));
    VSR_TRY(make_pair_maps(&c->WC_b, 128)); VSR_TRY(make_pair_maps(&c->WD_b, 128)); VSR_TRY(make_pair_maps(&c->WE_b, 96));
  }
  // the once-per-batch prologue GEMMs (U, U2, att_va projection) keep all three passes in fp16
  VSR_TRY(alloc_pair(c, &c->WU_b, c->NA, c->Fp, 128, PAIR_F16X3, true)); VSR_TRY(alloc_pair(c, &c->Wva_b, c->NVA, c->Fp, 128, PAIR_F16X3, true));
  if (d->img_second_lstm) VSR_TRY(alloc_pair(c, &c->WU2_b, c->ND, c->Fp, 128, PAIR_F16X3, true));
  VSR_TRY(pack_weights(c, w, 0));
  VSR_CHECK_CUDA(cudaStreamSynchronize(0));
  return VSR_OK;
}

static void drop_graphs(Ctx* c) {
  for (auto& g : c->graphs) cudaGraphExecDestroy(g.exec);
  c->graphs.clear();
  c->graph_seen.clear();
}

// The steps of a beam search through the graph cache: first sighting of a key runs eagerly, the second captures
// the same enqueue sequence on the library's capture stream and instantiates it, later ones replay it on `st`.
// A launch sequence through the graph cache: first sighting of a key runs eagerly, the second captures the same
// enqueue sequence on the library's capture stream and instantiates it, later ones replay it on `st`.
template <typename Enqueue>
static int run_graphed(Ctx* c, const Ctx::GraphKey& key, cudaStream_t st, Enqueue enqueue) {
  if (!c->graphs.empty() && c->graphs[0].key.epoch != c->epoch) drop_graphs(c);   // buffers moved: all stale
  ++c->graph_clock;
  for (auto& g : c->graphs)
    if (memcmp(&g.key, &key, sizeof(key)) == 0) {
      VSR_CHECK_CUDA(cudaGraphLaunch(g.exec, st));
      c->launches += g.launches; g.last_use = c->graph_clock;
      return VSR_OK;
    }
  bool seen = false;
  for (auto& s : c->graph_seen) seen = seen || memcmp(&s, &key, sizeof(key)) == 0;
  if (!seen) {
    if (c->graph_seen.size() >= 32) c->graph_seen.erase(c->graph_seen.begin());
    c->graph_seen.push_back(key);
    return enqueue(st);
  }
  if (c->cap_stream == nullptr) VSR_CHECK_CUDA(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
  const int64_t l0 = c->launches;
  VSR_CHECK_CUDA(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
  const int rc = enqueue(c->cap_stream);
  cudaGraph_t graph = nullptr;
  const cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
  const int64_t n_launch = c->launches - l0;
  c->launches = l0;
  if (rc != VSR_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
  VSR_CHECK_CUDA(ce);
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  VSR_CHECK_CUDA(ie);
  if (c->graphs.size() >= 16) {     // evict the least recently used
    size_t lru = 0;
    for (size_t i = 1; i < c->graphs.size(); ++i) if (c->graphs[i].last_use < c->graphs[lru].last_use) lru = i;
    cudaGraphExecDestroy(c->graphs[lru].exec);
    c->graphs.erase(c->graphs.begin() + lru);
  }
  c->graphs.push_back({key, exec, n_launch, c->graph_clock});
  VSR_CHECK_CUDA(cudaGraphLaunch(exec, st));
  c->launches += n_launch;
  return VSR_OK;
}

static Ctx::GraphKey graph_key(const Ctx* c, int kind) {
  Ctx::GraphKey key;
  memset(&key, 0, sizeof(key));
  key.kind = kind;
  key.epoch = c->epoch; key.det = c->det; key.det_seqs = c->det_seqs; key.slot_index = c->slot_index; key.verbs = c->verbs;
  key.det_stride = c->det_stride;
  key.b = c->b; key.D = c->D; key.L = c->L; key.R = c->R; key.n_img = c->n_img; key.verbs_dtype = c->verbs_dtype;
  key.feat_dtype = c->feat_dtype;   // the same addresses and shapes in another dtype run other kernels
  return key;
}

static bool graphs_usable(Ctx* c, cudaStream_t st) {
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) { cudaGetLastError(); cap = cudaStreamCaptureStatusActive; }
  return c->use_graphs && !c->profiling && cap == cudaStreamCaptureStatusNone;
}

static int prologue_impl(Ctx* c, const void* det, int64_t det_stride, int D, const void* det_seqs,
                         const int32_t* slot_index, int b, int L, int R, int feat_dtype, const void* verbs,
                         int verbs_dtype, cudaStream_t st) {
  VSR_REQUIRE(det != nullptr && (det_seqs != nullptr || slot_index != nullptr), VSR_EINVAL, "vsr_prologue: null input");
  VSR_REQUIRE(b > 0 && D > 0 && L > 0 && R > 0, VSR_EINVAL, "vsr_prologue: bad shape b=%d D=%d L=%d R=%d", b, D, L, R);
  VSR_REQUIRE(R <= 64, VSR_EINVAL, "vsr_prologue: R=%d regions per slot > 64 unsupported", R);
  VSR_REQUIRE(det_stride == 0 || det_stride >= (int64_t)D * c->F, VSR_EINVAL, "vsr_prologue: bad det_batch_stride");
  VSR_REQUIRE(verbs == nullptr || (verbs_dtype >= 0 && verbs_dtype <= 2), VSR_EINVAL, "vsr_prologue: bad verbs dtype");
  VSR_REQUIRE(slot_index == nullptr || det_stride == 0 || det_stride == (int64_t)D * c->F, VSR_EINVAL,
              "vsr_prologue_indexed: detections must be dense (b, D, F) or one shared image");
  const int esz = feat_elem_size(feat_dtype);
  VSR_REQUIRE(esz != 0, VSR_EINVAL, "vsr_prologue: feat_dtype=%d is not VSR_DT_F32, VSR_DT_F16 or VSR_DT_BF16", feat_dtype);
  VSR_REQUIRE(feat_dtype == VSR_DT_F32 || c->use_tc, VSR_EINVAL,
              "vsr_prologue: half-precision features need the tensor-core GEMMs; the fp32 FFMA twin (VSRDEC_GEMM=simt) "
              "reads features in place and takes fp32 only");
  // feature loads are four elements wide: 16 bytes in fp32, 8 in half precision
  VSR_REQUIRE(((uintptr_t)det % (4 * esz)) == 0 && ((uintptr_t)det_seqs % (4 * esz)) == 0 && (det_stride % 4) == 0,
              VSR_EINVAL, "vsr_prologue: feature tensors must be %d-byte aligned", 4 * esz);
  c->have_prologue = false;
  if (c->profiling) reset_phases(c);   // a decode job starts here
  c->b = b; c->D = D; c->L = L; c->R = R;
  c->n_img = det_stride == 0 ? 1 : b;
  c->det_seqs = det_seqs; c->slot_index = slot_index; c->det = det; c->det_stride = det_stride;
  c->feat_dtype = feat_dtype;
  c->verbs = verbs; c->verbs_dtype = verbs_dtype;
  const size_t n_img_pad = round_up(c->n_img, MPAD);
  if (n_img_pad > c->cap_img) {
    dev_free(c, c->img); dev_free(c, c->U); dev_free(c, c->U2);
    c->img = c->U = c->U2 = nullptr; c->cap_img = 0;
    ALLOC_F(c->img, n_img_pad * c->Fp); ALLOC_F(c->U, n_img_pad * c->NA);
    if (c->d.img_second_lstm) ALLOC_F(c->U2, n_img_pad * c->ND);
    VSR_TRY(alloc_pair(c, &c->img_b, (int)n_img_pad, c->Fp, MPAD, PAIR_F16X3));
    c->cap_img = n_img_pad;
  }
  // rows of the projection buffer: one per slot row (materialised form) or one per detection row plus one
  // per image, each block padded to whole 128-row tiles (index form)
  const size_t prow = slot_index == nullptr
                          ? (size_t)b * L * R
                          : (size_t)round_up(c->n_img * D, MPAD) + round_up(c->n_img, MPAD);
  if (prow > c->cap_P || (size_t)b * L + 1 > c->cap_slots) {
    const size_t need_rows = std::max(prow, c->cap_P), need_slots = std::max((size_t)b * L + 1, c->cap_slots);
    dev_free(c, c->P); dev_free(c, c->seq_valid); dev_free(c, c->slot_mask); dev_free(c, c->slot_base); dev_free(c, c->comp_valid);
    c->P = nullptr; c->seq_valid = nullptr; c->slot_mask = nullptr; c->slot_base = nullptr; c->comp_valid = nullptr;
    c->cap_P = 0; c->cap_slots = 0;
    ALLOC_F(c->P, round_up((int)need_rows, MPAD) * (size_t)c->NVA);
    VSR_TRY(dev_alloc(c, (void**)&c->seq_valid, round_up((int)need_rows, MPAD)));
    VSR_TRY(dev_alloc(c, (void**)&c->slot_mask, sizeof(unsigned long long) * need_slots));
    VSR_TRY(dev_alloc(c, (void**)&c->slot_base, sizeof(int32_t) * need_slots));
    VSR_TRY(dev_alloc(c, (void**)&c->comp_valid, round_up((int)need_rows, MPAD)));
    VSR_TRY(alloc_pair(c, &c->ds_b, round_up((int)need_rows, MPAD), c->Fp, MPAD, PAIR_F16X3));
    c->cap_P = need_rows; c->cap_slots = need_slots;
  }
  c->Pmean = slot_index != nullptr ? c->P + (size_t)round_up(c->n_img * D, MPAD) * c->NVA : nullptr;
  const size_t dvr = (size_t)c->n_img * D;
  if (dvr > c->cap_detv) {
    dev_free(c, c->det_valid); c->det_valid = nullptr; c->cap_detv = 0;
    VSR_TRY(dev_alloc(c, (void**)&c->det_valid, dvr));
    c->cap_detv = dvr;
  }
  VSR_TRY(ensure_rows(c, b));
  c->p_compact = slot_index == nullptr && c->use_tc;    // materialised slots on tensor cores: only valid rows are projected
  // the prologue's launch sequence goes through the same graph cache as the steps (kind 1)
  auto enqueue = [&](cudaStream_t s) {
    return slot_index == nullptr ? run_prologue(c, det, det_stride, s) : run_prologue_indexed(c, det, det_stride, s);
  };
  if (graphs_usable(c, st)) VSR_TRY(run_graphed(c, graph_key(c, 1), st, enqueue));
  else VSR_TRY(enqueue(st));
  c->have_prologue = true;
  return VSR_OK;
}

// dst[n][0:w] = src[n][0:w] with different leading dims
__global__ void k_copy2d(float* dst, int ld_dst, const float* src, int ld_src, int w, int rows) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (i < w && n < rows) dst[(size_t)n * ld_dst + i] = src[(size_t)n * ld_src + i];
}
__global__ void k_slots_from_i64(int32_t* ptr, const int64_t* slot, int rows, int L) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= rows) return;
  int64_t s = slot[n];
  s = s < 0 ? 0 : (s > L - 1 ? L - 1 : s);
  ptr[n] = (int32_t)s;
}
__global__ void k_fill_i32(int32_t* p, int v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

static int copy2d(Ctx* c, float* dst, int ld_dst, const float* src, int ld_src, int w, int rows, cudaStream_t st) {
  dim3 grid((w + 255) / 256, rows);
  k_copy2d<<<grid, 256, 0, st>>>(dst, ld_dst, src, ld_src, w, rows);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  return VSR_OK;
}

static int step_impl(Ctx* c, const float* h1, const float* c1, const float* h2, const float* c2,
                     const int64_t* slot, const int64_t* word, int use_verbs, int gt, float* h1o, float* c1o,
                     float* h2o, float* c2o, float* out_logp, float* gate_logp, cudaStream_t st) {
  VSR_REQUIRE(c->have_prologue, VSR_ESTATE, "vsr_step: call vsr_prologue first");
  VSR_REQUIRE(h1 && c1 && h2 && c2 && slot && word, VSR_EINVAL, "vsr_step: null state input");
  VSR_REQUIRE(!use_verbs || c->verbs != nullptr, VSR_EINVAL, "vsr_step: use_verbs without a verbs tensor");
  const int b = c->b, H = c->H;
  VSR_TRY(copy2d(c, c->h1, c->Hp, h1, H, H, b, st));
  VSR_TRY(copy2d(c, c->c1, c->Hp, c1, H, H, b, st));
  VSR_TRY(copy2d(c, c->h2, c->Hp, h2, H, H, b, st));
  VSR_TRY(copy2d(c, c->c2, c->Hp, c2, H, H, b, st));
  k_slots_from_i64<<<(b + 127) / 128, 128, 0, st>>>(c->ptr, slot, b, c->L);
  VSR_CHECK_CUDA(cudaGetLastError()); c->launches++;
  VSR_TRY(launch_words(c, word, b, st));
  if (c->use_tc) {
    VSR_TRY(launch_split_pair(c->h1, c->h1_b, (size_t)b * c->Hp, st));
    VSR_TRY(launch_split_pair(c->h2, c->h2_b, (size_t)b * c->Hp, st));
    c->launches += 2;
  }
  StepIO io{};
  io.rows = b; io.cur_beam = 1; io.use_verbs = use_verbs != 0; io.gt = gt != 0;
  io.out_logp = out_logp; io.out_stride = c->V; io.gate_out = gate_logp; io.gate_stride = 2; io.topk = 0;
  io.need_h32 = true;
  VSR_TRY(run_step(c, io, st));
  if (h1o) VSR_TRY(copy2d(c, h1o, H, c->h1n, c->Hp, H, b, st));
  if (c1o) VSR_TRY(copy2d(c, c1o, H, c->c1n, c->Hp, H, b, st));
  if (h2o) VSR_TRY(copy2d(c, h2o, H, c->h2n, c->Hp, H, b, st));
  if (c2o) VSR_TRY(copy2d(c, c2o, H, c->c2n, c->Hp, H, b, st));
  return VSR_OK;
}

// state init + T x (decoder step, beam selection + reorder): everything of a beam search except the back-track
static int enqueue_beam_steps(Ctx* c, int k, const int64_t* eos, int use_verbs, int gt, const VsrTrace* tr,
                              cudaStream_t st) {
  const int b = c->b, T = c->d.seq_len;
  VSR_TRY(launch_state_init(c, b, st));
  const bool have_forced = tr && tr->forced_beam && tr->forced_word && tr->forced_gate;
  if (c->profiling) {          // per-step latency: one event before every step and one after the last
    for (cudaEvent_t e : c->step_ev) cudaEventDestroy(e);
    c->step_ev.clear();
  }
  for (int t = 0; t < T; ++t) {
    if (c->profiling) {
      cudaEvent_t e;
      if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); c->step_ev.push_back(e); }
    }
    const int cur = t == 0 ? 1 : k;
    const int rows = b * cur;
    StepIO io{};
    io.rows = rows; io.cur_beam = cur; io.use_verbs = use_verbs != 0; io.gt = gt != 0; io.topk = k;
    io.zero_state = t == 0;
    io.ngram_block = c->ngram > 0; io.t = t;
    if (tr && tr->step_out) { io.out_logp = tr->step_out + (size_t)t * b * k * c->V; io.out_stride = c->V; }
    if (tr && tr->step_gate) { io.gate_out = tr->step_gate + (size_t)t * b * k * 2; io.gate_stride = 2; }
    attn_step_io(c, io, t, (int64_t)b * k);
    VSR_TRY(run_step(c, io, st));
    const size_t fo = (size_t)t * b * k;
    VSR_TRY(launch_beam_step(c, t, b, cur, k, eos[0], eos[1], have_forced ? tr->forced_beam + fo : nullptr,
                             have_forced ? tr->forced_word + fo : nullptr,
                             have_forced ? tr->forced_gate + fo : nullptr, t + 1 < T, st));
  }
  if (c->profiling) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) == cudaSuccess) { cudaEventRecord(e, st); c->step_ev.push_back(e); }
  }
  return VSR_OK;
}

// the steps of a beam search (kind 0)
static int beam_steps_graphed(Ctx* c, int k, const int64_t* eos, int use_verbs, int gt, cudaStream_t st) {
  Ctx::GraphKey key = graph_key(c, 0);
  key.eos0 = eos[0]; key.eos1 = eos[1];
  key.k = k; key.use_verbs = use_verbs; key.gt = gt; key.T = c->d.seq_len; key.attn = c->attn_capture;
  key.ngram = c->ngram;
  if (c->beam_groups > 1) { key.beam_groups = c->beam_groups; memcpy(&key.beam_penalty, &c->beam_penalty, 4); }
  return run_graphed(c, key, st, [&](cudaStream_t s) { return enqueue_beam_steps(c, k, eos, use_verbs, gt, nullptr, s); });
}

static int beam_search_impl(Ctx* c, int k, int out_size, const int64_t* eos, int use_verbs, int gt,
                            int64_t* out_words, int64_t* out_gates, float* lp_words, float* lp_gates,
                            const VsrTrace* tr, cudaStream_t st) {
  VSR_REQUIRE(c->have_prologue, VSR_ESTATE, "vsr_beam_search: call vsr_prologue first");
  VSR_REQUIRE(k >= 1 && k <= VSR_MAX_BEAM, VSR_EINVAL, "vsr_beam_search: beam_size=%d not in [1,%d]", k, VSR_MAX_BEAM);
  VSR_REQUIRE(out_size >= 1 && out_size <= k, VSR_EINVAL, "vsr_beam_search: out_size=%d not in [1,beam]", out_size);
  VSR_REQUIRE(c->V >= k, VSR_EINVAL, "vsr_beam_search: vocabulary (%d) smaller than the beam (%d): a row has fewer than "
              "beam distinct word candidates", c->V, k);
  VSR_REQUIRE(c->d.seq_len <= VSR_MAX_SEQ_LEN, VSR_EINVAL, "vsr_beam_search: seq_len=%d > %d unsupported by the back-track kernel",
              c->d.seq_len, VSR_MAX_SEQ_LEN);
  VSR_REQUIRE(eos && out_words && out_gates && lp_words && lp_gates, VSR_EINVAL, "vsr_beam_search: null argument");
  VSR_REQUIRE(!use_verbs || c->verbs != nullptr, VSR_EINVAL, "vsr_beam_search: use_verbs without a verbs tensor");
  const int b = c->b, T = c->d.seq_len;
  VSR_REQUIRE(c->ngram == 0 || c->V >= k + T - 1, VSR_EINVAL, "vsr_beam_search: n-gram blocking needs vocab_size (%d) >= "
              "beam + seq_len - 1 (%d), so that every row keeps beam words that are not banned", c->V, k + T - 1);
  VSR_REQUIRE(k % c->beam_groups == 0, VSR_EINVAL, "vsr_beam_search: beam_size=%d is not a multiple of the %d beam groups "
              "(vsr_set_beam_diversity)", k, c->beam_groups);
  VSR_TRY(ensure_rows(c, b * k));
  if (c->ngram > 0) VSR_TRY(ensure_whist(c, b * k));
  VSR_TRY(ensure_beam_ws(c, b, T));
  VSR_TRY(attn_begin(c, (int64_t)b * k, T, (size_t)b * out_size * T));
  c->hist_T = T; c->hist_b = b; c->hist_k = k;
  // graph replay unless a trace is requested, the phase profiler is on, or the caller is capturing itself
  if (tr == nullptr && graphs_usable(c, st))
    VSR_TRY(beam_steps_graphed(c, k, eos, use_verbs, gt, st));
  else
    VSR_TRY(enqueue_beam_steps(c, k, eos, use_verbs, gt, tr, st));
  VSR_TRY(launch_backtrack(c, b, k, T, out_size, out_words, out_gates, lp_words, lp_gates,
                           c->attn_capture ? c->attn_path : nullptr, st));
  attn_done(c, true, T, b * out_size, (int64_t)b * k);
  return VSR_OK;
}

// (re)size the all-steps buffers of the batched teacher-forced forward
static int ensure_fwd_ws(Ctx* c, int rows) {
  if (rows <= c->cap_fwd_rows) return VSR_OK;
  const int cap = round_up(rows, MPAD);
  dev_free(c, c->logits_all); dev_free(c, c->gate_all);
  c->logits_all = c->gate_all = nullptr; c->cap_fwd_rows = 0;
  ALLOC_F(c->logits_all, (size_t)cap * c->NE); ALLOC_F(c->gate_all, (size_t)cap * 2);
  VSR_TRY(alloc_pair(c, &c->h2all_b, cap, c->Hp, MPAD, step_kind(c)));
  c->cap_fwd_rows = cap;
  return VSR_OK;
}

// the recurrent part of the teacher-forced unroll: everything except the vocabulary projection, which does not feed
// back (CaptioningModel.py:22-36) and therefore runs ONCE over all (caption, step) rows after the loop
static int enqueue_forward_steps(Ctx* c, const int64_t* captions, int T, bool batched, float* out, float* gate, cudaStream_t st) {
  const int b = c->b;
  VSR_TRY(launch_state_init(c, b, st));
  // the first input token is captions[:, 0], not bos (controllable_captioning.py:131-133)
  for (int t = 0; t < T; ++t) {
    if (t == 0) {
      // xt <- embed[captions[:,0]], slot 0
      VSR_CHECK_CUDA(cudaMemcpy2DAsync(c->word_in, sizeof(int64_t), captions, sizeof(int64_t) * T,
                                       sizeof(int64_t), b, cudaMemcpyDeviceToDevice, st));
      VSR_TRY(launch_words(c, c->word_in, b, st));
    }
    StepIO io{};
    io.rows = b; io.cur_beam = 1; io.use_verbs = false; io.gt = false; io.topk = 0;
    io.zero_state = t == 0;
    attn_step_io(c, io, t, b);
    if (batched) {
      io.skip_vocab = true;
      VSR_TRY(run_step(c, io, st));
      VSR_TRY(launch_gate_head(c, b, c->gate_all + (size_t)t * 2, (int64_t)T * 2, st));      // row i -> (i, t)
      VSR_TRY(launch_rows_to_all(c, c->h2n_b, c->h2all_b, b, T, t, st));
    } else {
      io.out_logp = out + (size_t)t * c->V; io.out_stride = (int64_t)T * c->V;
      io.gate_out = gate + (size_t)t * 2; io.gate_stride = (int64_t)T * 2;
      VSR_TRY(run_step(c, io, st));
    }
    if (t + 1 < T) VSR_TRY(launch_commit_identity(c, b, captions + (t + 1), T, t + 1, -1, st));
  }
  if (batched) VSR_TRY(run_vocab_rows(c, c->h2all_b, c->logits_all, b * T, nullptr, st, false));   // M = b*T rows
  return VSR_OK;
}

static int forward_impl(Ctx* c, const int64_t* captions, int T, float* out, float* gate, cudaStream_t st) {
  VSR_REQUIRE(c->have_prologue, VSR_ESTATE, "vsr_forward_teacher: call vsr_prologue first");
  VSR_REQUIRE(captions && out && gate, VSR_EINVAL, "vsr_forward_teacher: null argument");
  VSR_REQUIRE(T >= 1 && T <= c->L, VSR_EINVAL, "vsr_forward_teacher: T=%d exceeds the prologue's slot count L=%d", T, c->L);
  const int b = c->b;
  VSR_TRY(ensure_rows(c, b));
  VSR_TRY(attn_begin(c, b, T, 0));
  const bool batched = c->use_tc;        // (the FFMA twin keeps the plain per-step unroll)
  if (!batched) {
    VSR_TRY(enqueue_forward_steps(c, captions, T, false, out, gate, st));
    attn_done(c, false, T, b, b);
    return VSR_OK;
  }
  VSR_TRY(ensure_fwd_ws(c, b * T));
  if (graphs_usable(c, st)) {            // the loop + the batched vocabulary GEMM replay from the graph cache (kind 2)
    Ctx::GraphKey key = graph_key(c, 2);
    key.captions = captions; key.T = T; key.attn = c->attn_capture;
    VSR_TRY(run_graphed(c, key, st, [&](cudaStream_t s) { return enqueue_forward_steps(c, captions, T, true, nullptr, nullptr, s); }));
  } else {
    VSR_TRY(enqueue_forward_steps(c, captions, T, true, nullptr, nullptr, st));
  }
  // caller-owned outputs are written outside the graph: log-softmax of the b*T vocabulary rows, and the gate rows
  VSR_TRY(run_vocab_rows(c, c->h2all_b, c->logits_all, b * T, out, st, true));
  VSR_CHECK_CUDA(cudaMemcpyAsync(gate, c->gate_all, sizeof(float) * (size_t)b * T * 2, cudaMemcpyDeviceToDevice, st));
  attn_done(c, false, T, b, b);
  return VSR_OK;
}

static int greedy_impl(Ctx* c, int64_t* out_words, int64_t* out_gates, cudaStream_t st) {
  VSR_REQUIRE(c->have_prologue, VSR_ESTATE, "vsr_greedy: call vsr_prologue first");
  VSR_REQUIRE(out_words && out_gates, VSR_EINVAL, "vsr_greedy: null argument");
  const int b = c->b, T = c->d.seq_len;
  VSR_REQUIRE(c->ngram == 0 || c->V >= T, VSR_EINVAL, "vsr_greedy: n-gram blocking needs vocab_size (%d) >= seq_len (%d)",
              c->V, T);
  VSR_TRY(ensure_rows(c, b));
  if (c->ngram > 0) VSR_TRY(ensure_whist(c, b));
  VSR_TRY(ensure_beam_ws(c, b, T));
  VSR_TRY(attn_begin(c, b, T, 0));
  VSR_TRY(launch_state_init(c, b, st));
  for (int t = 0; t < T; ++t) {
    StepIO io{};
    io.rows = b; io.cur_beam = 1; io.use_verbs = false; io.gt = false; io.topk = 1;
    io.zero_state = t == 0;
    io.ngram_block = c->ngram > 0; io.t = t;
    attn_step_io(c, io, t, b);
    VSR_TRY(run_step(c, io, st));
    VSR_TRY(launch_greedy_pick(c, b, t, T, out_words, out_gates, st));
    if (t + 1 < T) VSR_TRY(launch_commit_identity(c, b, nullptr, 0, -1, c->ngram > 0 ? t : -1, st));
  }
  attn_done(c, false, T, b, b);
  return VSR_OK;
}

// multinomial sampling decode: the whole loop on the device, one pick kernel per step, no host work in between.
// p.n draws per caption run as rows = b * p.n with cur_beam = p.n: every row starts from init_state, statics are read by
// caption = row / p.n, and the draws of a row depend on (seed, caption, draw, step) only (vsr_sample_ex in vsrdec.h).
static int sample_impl(Ctx* c, const VsrSampleParams& p, int64_t* out_words, int64_t* out_gates, float* lp_words,
                       float* lp_gates, cudaStream_t st) {
  VSR_REQUIRE(c->have_prologue, VSR_ESTATE, "vsr_sample: call vsr_prologue first");
  VSR_REQUIRE(out_words && out_gates && lp_words && lp_gates, VSR_EINVAL, "vsr_sample: null argument");
  VSR_REQUIRE(p.n >= 1, VSR_EINVAL, "vsr_sample_ex: n=%d draws per caption, must be >= 1", p.n);
  VSR_REQUIRE(isfinite(p.temperature) && p.temperature > 0.f, VSR_EINVAL,
              "vsr_sample_ex: temperature=%g must be finite and > 0", (double)p.temperature);
  VSR_REQUIRE(p.top_k >= 0, VSR_EINVAL, "vsr_sample_ex: top_k=%d must be >= 0 (0 = off)", p.top_k);
  VSR_REQUIRE(p.top_p > 0.f && p.top_p <= 1.f, VSR_EINVAL, "vsr_sample_ex: top_p=%g not in (0, 1]", (double)p.top_p);
  VSR_REQUIRE(!p.use_verbs || c->verbs != nullptr, VSR_EINVAL, "vsr_sample_ex: use_verbs without a verbs tensor");
  const int b = c->b, T = c->d.seq_len;
  VSR_REQUIRE((int64_t)b * p.n <= (int64_t)1 << 30, VSR_EINVAL, "vsr_sample_ex: b*n = %lld rows > 2^30 unsupported",
              (long long)b * p.n);
  VSR_REQUIRE(c->ngram == 0 || c->V >= T, VSR_EINVAL, "vsr_sample_ex: n-gram blocking needs vocab_size (%d) >= seq_len (%d)",
              c->V, T);
  const int rows = b * p.n;
  VSR_TRY(ensure_rows(c, rows));
  VSR_TRY(ensure_sel(c, rows));
  if (c->ngram > 0) VSR_TRY(ensure_whist(c, rows));
  VSR_TRY(attn_begin(c, rows, T, 0));
  VSR_TRY(launch_state_init(c, rows, st));
  for (int t = 0; t < T; ++t) {
    StepIO io{};
    io.rows = rows; io.cur_beam = p.n; io.use_verbs = p.use_verbs != 0; io.gt = p.gt != 0;
    io.topk = 0;     // statistics + gate head (+ forced word) only
    io.zero_state = t == 0;
    attn_step_io(c, io, t, rows);
    VSR_TRY(run_step(c, io, st));
    VSR_TRY(launch_sample_pick(c, rows, t, T, p, out_words, out_gates, lp_words, lp_gates, st));
    if (t + 1 < T) VSR_TRY(launch_commit_identity(c, rows, nullptr, 0, -1, c->ngram > 0 ? t : -1, st));
  }
  attn_done(c, false, T, rows, rows);
  return VSR_OK;
}

}  // namespace vsr

// ============================================================================ C ABI
using vsr::Ctx;

// Every entry point runs on the handle's device regardless of the caller's current device (restored on return).
struct DeviceGuard {
  int prev = -1; bool switched = false;
  explicit DeviceGuard(const vsr::Ctx* c) {
    if (c != nullptr && cudaGetDevice(&prev) == cudaSuccess && prev != c->device) switched = cudaSetDevice(c->device) == cudaSuccess;
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

extern "C" {

const char* vsr_last_error(void) { return vsr::g_err; }
int32_t vsr_abi_version(void) { return VSR_ABI_VERSION; }

int vsr_create(const VsrDims* dims, const float* const* weights, vsr_handle* out) {
  if (out == nullptr) { vsr::set_error("vsr_create: null out"); return VSR_EINVAL; }
  *out = nullptr;
  Ctx* c = nullptr;
  const int r = vsr::create_impl(dims, weights, &c);
  if (r != VSR_OK) { if (c) vsr_destroy((vsr_handle)c); return r; }
  *out = (vsr_handle)c;
  return VSR_OK;
}

int vsr_load_weights(vsr_handle h, const float* const* weights, void* stream) {
  if (!h || !weights) { vsr::set_error("vsr_load_weights: null argument"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  // the hoisted projections (U / U2 / P / img) were made with the old att_va / W_ih: the prologue must be re-run
  ((Ctx*)h)->have_prologue = false;
  return vsr::pack_weights((Ctx*)h, weights, (cudaStream_t)stream);
}

void vsr_destroy(vsr_handle h) {
  if (!h) return;
  Ctx* c = (Ctx*)h;
  DeviceGuard dg(c);
  cudaDeviceSynchronize();
  vsr::reset_phases(c);
  for (cudaEvent_t e : c->step_ev) cudaEventDestroy(e);
  vsr::drop_graphs(c);
  if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
  for (void* p : c->owned) cudaFree(p);
  delete c;
}

int vsr_set_verb_table(vsr_handle h, const int64_t* keys, const int32_t* offsets, const int32_t* vocab_idx,
                       int32_t n_keys) {
  if (!h) { vsr::set_error("vsr_set_verb_table: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  Ctx* c = (Ctx*)h;
  VSR_CHECK_CUDA(cudaDeviceSynchronize());
  vsr::dev_free(c, c->vt_keys); vsr::dev_free(c, c->vt_off); vsr::dev_free(c, c->vt_idx);
  c->vt_keys = nullptr; c->vt_off = nullptr; c->vt_idx = nullptr; c->vt_n = 0;
  if (n_keys <= 0) return VSR_OK;
  VSR_REQUIRE(keys && offsets && vocab_idx, VSR_EINVAL, "vsr_set_verb_table: null table");
  for (int i = 1; i < n_keys; ++i)
    VSR_REQUIRE(keys[i] > keys[i - 1], VSR_EINVAL, "vsr_set_verb_table: keys must be strictly increasing");
  VSR_REQUIRE(offsets[0] == 0, VSR_EINVAL, "vsr_set_verb_table: offsets[0] must be 0");
  for (int i = 0; i < n_keys; ++i)
    VSR_REQUIRE(offsets[i + 1] >= offsets[i], VSR_EINVAL, "vsr_set_verb_table: offsets must be non-decreasing");
  const int nnz = offsets[n_keys];
  for (int i = 0; i < nnz; ++i)
    VSR_REQUIRE(vocab_idx[i] >= 0 && vocab_idx[i] < c->V, VSR_EINVAL, "vsr_set_verb_table: vocab index %d out of range", vocab_idx[i]);
  VSR_TRY(vsr::dev_alloc(c, (void**)&c->vt_keys, sizeof(int64_t) * n_keys, false));
  VSR_TRY(vsr::dev_alloc(c, (void**)&c->vt_off, sizeof(int32_t) * (n_keys + 1), false));
  VSR_TRY(vsr::dev_alloc(c, (void**)&c->vt_idx, sizeof(int32_t) * std::max(nnz, 1), false));
  VSR_CHECK_CUDA(cudaMemcpy(c->vt_keys, keys, sizeof(int64_t) * n_keys, cudaMemcpyHostToDevice));
  VSR_CHECK_CUDA(cudaMemcpy(c->vt_off, offsets, sizeof(int32_t) * (n_keys + 1), cudaMemcpyHostToDevice));
  if (nnz > 0) VSR_CHECK_CUDA(cudaMemcpy(c->vt_idx, vocab_idx, sizeof(int32_t) * nnz, cudaMemcpyHostToDevice));
  c->vt_n = n_keys;
  return VSR_OK;
}

int vsr_prologue_ex(vsr_handle h, const void* det, int64_t det_batch_stride, int32_t D, const void* det_seqs,
                    int32_t b, int32_t L, int32_t R, int32_t feat_dtype, const void* verbs, int32_t verbs_dtype,
                    void* stream) {
  if (!h) { vsr::set_error("vsr_prologue: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::prologue_impl((Ctx*)h, det, det_batch_stride, D, det_seqs, nullptr, b, L, R, feat_dtype, verbs,
                            verbs_dtype, (cudaStream_t)stream);
}

int vsr_prologue_indexed_ex(vsr_handle h, const void* det, int64_t det_batch_stride, int32_t D,
                            const int32_t* slot_index, int32_t b, int32_t L, int32_t R, int32_t feat_dtype,
                            const void* verbs, int32_t verbs_dtype, void* stream) {
  if (!h || !slot_index) { vsr::set_error("vsr_prologue_indexed: null argument"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::prologue_impl((Ctx*)h, det, det_batch_stride, D, nullptr, slot_index, b, L, R, feat_dtype, verbs,
                            verbs_dtype, (cudaStream_t)stream);
}

int vsr_prologue(vsr_handle h, const float* det, int64_t det_batch_stride, int32_t D, const float* det_seqs,
                 int32_t b, int32_t L, int32_t R, const void* verbs, int32_t verbs_dtype, void* stream) {
  return vsr_prologue_ex(h, det, det_batch_stride, D, det_seqs, b, L, R, VSR_DT_F32, verbs, verbs_dtype, stream);
}

int vsr_prologue_indexed(vsr_handle h, const float* det, int64_t det_batch_stride, int32_t D,
                         const int32_t* slot_index, int32_t b, int32_t L, int32_t R, const void* verbs,
                         int32_t verbs_dtype, void* stream) {
  return vsr_prologue_indexed_ex(h, det, det_batch_stride, D, slot_index, b, L, R, VSR_DT_F32, verbs, verbs_dtype,
                                 stream);
}

int vsr_step(vsr_handle h, const float* h1, const float* c1, const float* h2, const float* c2,
             const int64_t* slot, const int64_t* word, int32_t use_verbs, int32_t gt, float* h1o, float* c1o,
             float* h2o, float* c2o, float* out_logp, float* gate_logp, void* stream) {
  if (!h) { vsr::set_error("vsr_step: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::step_impl((Ctx*)h, h1, c1, h2, c2, slot, word, use_verbs, gt, h1o, c1o, h2o, c2o, out_logp,
                        gate_logp, (cudaStream_t)stream);
}

int vsr_beam_search(vsr_handle h, int32_t beam_size, int32_t out_size, const int64_t* eos_idxs,
                    int32_t use_verbs, int32_t gt, int64_t* out_words, int64_t* out_gates, float* lp_words,
                    float* lp_gates, const VsrTrace* trace, void* stream) {
  if (!h) { vsr::set_error("vsr_beam_search: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::beam_search_impl((Ctx*)h, beam_size, out_size, eos_idxs, use_verbs, gt, out_words, out_gates,
                               lp_words, lp_gates, trace, (cudaStream_t)stream);
}

int vsr_get_history(vsr_handle h, int32_t* parent, int32_t* word, int32_t* gate, float* score, void* stream) {
  if (!h) { vsr::set_error("vsr_get_history: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  Ctx* c = (Ctx*)h;
  VSR_REQUIRE(c->hist_T > 0, VSR_ESTATE, "vsr_get_history: no beam search has run on this handle");
  const size_t n = (size_t)c->hist_T * c->hist_b * c->hist_k;
  cudaStream_t st = (cudaStream_t)stream;
  if (parent) VSR_CHECK_CUDA(cudaMemcpyAsync(parent, c->hist_parent, n * 4, cudaMemcpyDeviceToDevice, st));
  if (word) VSR_CHECK_CUDA(cudaMemcpyAsync(word, c->hist_word, n * 4, cudaMemcpyDeviceToDevice, st));
  if (gate) VSR_CHECK_CUDA(cudaMemcpyAsync(gate, c->hist_gate, n * 4, cudaMemcpyDeviceToDevice, st));
  if (score) VSR_CHECK_CUDA(cudaMemcpyAsync(score, c->hist_score, n * 4, cudaMemcpyDeviceToDevice, st));
  return VSR_OK;
}

int vsr_set_attention_capture(vsr_handle h, int32_t enabled) {
  if (!h) { vsr::set_error("vsr_set_attention_capture: null handle"); return VSR_EINVAL; }
  ((Ctx*)h)->attn_capture = enabled != 0;
  return VSR_OK;
}

int vsr_set_no_repeat_ngram(vsr_handle h, int32_t n) {
  if (!h) { vsr::set_error("vsr_set_no_repeat_ngram: null handle"); return VSR_EINVAL; }
  Ctx* c = (Ctx*)h;
  VSR_REQUIRE(n >= 0 && n <= c->d.seq_len, VSR_EINVAL, "vsr_set_no_repeat_ngram: n=%d not in [0, seq_len=%d] (0 = off)", n,
              c->d.seq_len);
  c->ngram = n;
  return VSR_OK;
}

int vsr_set_beam_diversity(vsr_handle h, int32_t groups, float penalty) {
  if (!h) { vsr::set_error("vsr_set_beam_diversity: null handle"); return VSR_EINVAL; }
  Ctx* c = (Ctx*)h;
  VSR_REQUIRE(groups >= 1 && groups <= VSR_MAX_BEAM, VSR_EINVAL, "vsr_set_beam_diversity: groups=%d not in [1, %d] (1 = off)",
              groups, VSR_MAX_BEAM);
  VSR_REQUIRE(isfinite(penalty) && penalty >= 0.f, VSR_EINVAL, "vsr_set_beam_diversity: penalty=%g is not finite and >= 0",
              (double)penalty);
  c->beam_groups = groups; c->beam_penalty = penalty;
  return VSR_OK;
}

int vsr_get_attention(vsr_handle h, float* alpha, int32_t* slot, void* stream) {
  if (!h) { vsr::set_error("vsr_get_attention: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  Ctx* c = (Ctx*)h;
  VSR_REQUIRE(c->attn_ready, VSR_ESTATE,
              "vsr_get_attention: the last decode on this handle ran without attention capture (vsr_set_attention_capture)");
  VSR_REQUIRE(alpha && slot, VSR_EINVAL, "vsr_get_attention: null argument");
  return vsr::launch_attn_gather(c, c->attn_beam ? c->attn_path : nullptr, c->attn_n_out, c->attn_T, alpha, slot,
                                 (cudaStream_t)stream);
}

int vsr_forward_teacher(vsr_handle h, const int64_t* captions, int32_t T, float* out, float* gate, void* stream) {
  if (!h) { vsr::set_error("vsr_forward_teacher: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::forward_impl((Ctx*)h, captions, T, out, gate, (cudaStream_t)stream);
}

int vsr_greedy(vsr_handle h, int64_t* out_words, int64_t* out_gates, void* stream) {
  if (!h) { vsr::set_error("vsr_greedy: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::greedy_impl((Ctx*)h, out_words, out_gates, (cudaStream_t)stream);
}

int vsr_sample_ex(vsr_handle h, const VsrSampleParams* p, int64_t* out_words, int64_t* out_gates, float* lp_words,
                  float* lp_gates, void* stream) {
  if (!h || !p) { vsr::set_error("vsr_sample_ex: null argument"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  return vsr::sample_impl((Ctx*)h, *p, out_words, out_gates, lp_words, lp_gates, (cudaStream_t)stream);
}

int vsr_sample(vsr_handle h, uint64_t seed, int64_t* out_words, int64_t* out_gates, float* lp_words, float* lp_gates,
               void* stream) {
  const VsrSampleParams p = {seed, 1, 1.f, 0, 1.f, 0, 0};
  return vsr_sample_ex(h, &p, out_words, out_gates, lp_words, lp_gates, stream);
}

int64_t vsr_launch_count(vsr_handle h) { return h ? ((Ctx*)h)->launches : -1; }

const char* vsr_gemm_kind(vsr_handle h) {
  if (!h) return "none";
  const Ctx* c = (const Ctx*)h;
  return !c->use_tc ? "simt-fp32" : (c->gemm_f8 ? "tcgen05-f16+f8x2" : "tcgen05-f16x3");
}

int vsr_set_profiling(vsr_handle h, int32_t enabled) {
  if (!h) { vsr::set_error("vsr_set_profiling: null handle"); return VSR_EINVAL; }
  Ctx* c = (Ctx*)h;
  c->profiling = enabled != 0;
  vsr::reset_phases(c);
  return VSR_OK;
}

int vsr_get_phase_times(vsr_handle h, const char** names, float* ms, int32_t* launches, int32_t cap) {
  if (!h) { vsr::set_error("vsr_get_phase_times: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  Ctx* c = (Ctx*)h;
  VSR_CHECK_CUDA(cudaDeviceSynchronize());
  int n = 0;
  for (int i = 0; i < vsr::PH_COUNT && n < cap; ++i) {
    float total = 0.f;
    const auto& ev = c->phases[i].ev;
    for (size_t j = 0; j + 1 < ev.size(); j += 2) {
      float t = 0.f;
      if (cudaEventElapsedTime(&t, ev[j], ev[j + 1]) == cudaSuccess) total += t;
    }
    if (names) names[n] = c->phases[i].name;
    if (ms) ms[n] = total;
    if (launches) launches[n] = c->phases[i].launches;
    ++n;
  }
  return n;
}

int vsr_get_step_times(vsr_handle h, float* ms, int32_t cap) {
  if (!h) { vsr::set_error("vsr_get_step_times: null handle"); return VSR_EINVAL; }
  DeviceGuard dg((const vsr::Ctx*)h);
  Ctx* c = (Ctx*)h;
  VSR_CHECK_CUDA(cudaDeviceSynchronize());
  int n = 0;
  for (size_t j = 0; j + 1 < c->step_ev.size() && n < cap; ++j, ++n) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, c->step_ev[j], c->step_ev[j + 1]) != cudaSuccess) t = -1.f;
    if (ms) ms[n] = t;
  }
  return n;
}

}  // extern "C"
