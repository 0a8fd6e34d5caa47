/*
 * vsrdec.h — C ABI of the B200-native role-shift captioning decoder (libvsrdec.so).
 *
 * The reference (mad-red/VSR-guided-CIC) has no FFI/plugin layer: its boundary for this
 * path is the Python class surface `ControllableCaptioningModel` / `CaptioningModel`
 * (models/controllable_captioning.py:10-303, models/CaptioningModel.py:8-294).  The
 * drop-in `models` package in this repo keeps that surface and forwards every hot call
 * to the entry points below through ctypes.  Each entry point cites the reference
 * interface it replaces.
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary;
 *   - unless marked [host], every pointer is a DEVICE pointer on the handle's device,
 *     fp32 tensors contiguous row-major, index tensors int64 (torch.long);
 *   - the library BORROWS caller pointers for the duration of a call only, except the
 *     inputs given to vsr_prologue(), which must stay alive and unchanged until the last
 *     decode call that uses that prologue has been enqueued AND executed (they are read
 *     by the step kernels);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream); no entry point synchronises the host with the device except
 *     vsr_create / vsr_destroy / vsr_set_verb_table;
 *   - every function returns 0 on success or a negative VSR_E* code; the message is
 *     available from vsr_last_error() (thread-local).  Nothing throws across the ABI;
 *   - there is NO CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef VSRDEC_H_
#define VSRDEC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSR_ABI_VERSION 1

#define VSR_OK 0
#define VSR_EINVAL (-1)  /* bad argument / unsupported size                       */
#define VSR_ECUDA (-2)   /* CUDA runtime error (message has the cudaError string) */
#define VSR_ENOMEM (-3)  /* device allocation failed                              */
#define VSR_ESTATE (-4)  /* call order violated (e.g. decode before prologue)     */

#define VSR_MAX_BEAM 8   /* largest beam_size supported by the fused top-k        */
#define VSR_MAX_SEQ_LEN 256 /* largest seq_len of the beam-search back-track kernel  */
#define VSR_NUM_WEIGHTS 28

/* dtype tags: the `verbs` tensor takes F64 / F32 / I64 (eval_coco.py:240 hands float64 from numpy);
 * the region features of vsr_prologue_ex / vsr_prologue_indexed_ex take F32 / F16 / BF16 */
#define VSR_DT_F64 0
#define VSR_DT_F32 1
#define VSR_DT_I64 2
#define VSR_DT_F16 3   /* IEEE binary16 (__half)      */
#define VSR_DT_BF16 4  /* bfloat16 (__nv_bfloat16)    */

typedef struct VsrHandle_* vsr_handle;

/* Constructor arguments of ControllableCaptioningModel (controllable_captioning.py:11-12). */
typedef struct VsrDims {
  int32_t seq_len;
  int32_t vocab_size;
  int32_t bos_idx;
  int32_t det_feat_size;       /* must be a multiple of 4 (four-element feature loads) */
  int32_t input_encoding_size;
  int32_t rnn_size;
  int32_t att_size;
  int32_t h2_first_lstm;       /* bool */
  int32_t img_second_lstm;     /* bool */
} VsrDims;

/* Optional per-step trace buffers (parity tests / trajectory replay).  Any pointer may be NULL.
 * Rows of step t are caption-major (row = caption*cur_beam + beam, cur_beam = 1 at t = 0). */
typedef struct VsrTrace {
  float* step_out;            /* [T][b*beam][V]  word log-probs returned by step t          */
  float* step_gate;           /* [T][b*beam][2]  gate log-probs returned by step t          */
  const int32_t* forced_beam; /* [T][b][beam]    replay these selections instead of top-k   */
  const int32_t* forced_word; /* [T][b][beam]                                               */
  const int32_t* forced_gate; /* [T][b][beam]                                               */
} VsrTrace;

const char* vsr_last_error(void);
int32_t vsr_abi_version(void);

/* Replaces ControllableCaptioningModel.__init__ + state_dict ownership
 * (controllable_captioning.py:11-70).  `weights` [host array of 28 device pointers] follows
 * the state_dict registration order:
 *   0 embed.weight (V,E)            1 W1_is.weight (H,in1)       2 W1_is.bias (H)
 *   3 W1_hs.weight (H,H)            4 W1_hs.bias (H)             5 att_va.weight (A,F)
 *   6 att_ha.weight (A,H)           7 att_a.weight (1,A)         8 att_sa.weight (A,H)
 *   9 att_s.weight (1,A)           10 lstm_cell_1.weight_ih (4H,in1)
 *  11 lstm_cell_1.weight_hh (4H,H) 12 lstm_cell_1.bias_ih (4H)  13 lstm_cell_1.bias_hh (4H)
 *  14 lstm_cell_2.weight_ih (4H,in2) 15 lstm_cell_2.weight_hh (4H,H)
 *  16 lstm_cell_2.bias_ih (4H)     17 lstm_cell_2.bias_hh (4H)  18 out_fc.weight (V,H)
 *  19 out_fc.bias (V)              20 s_fc.weight (F,H)         21 s_fc.bias (F)
 *  22 W1_ig.weight (H,in1)         23 W1_ig.bias (H)            24 W1_hg.weight (H,H)
 *  25 W1_hg.bias (H)               26 att_ga.weight (A,H)       27 att_g.weight (1,A)
 * with in1 = [H if h2_first_lstm] + F + E  (column order [h2 | img | xt], :228) and
 * in2 = H + F [+ F if img_second_lstm]     (column order [h1 | att | img], :254-257).
 * The library keeps its own packed (stacked / K-padded) copy; the caller keeps ownership
 * of the originals. */
int vsr_create(const VsrDims* dims, const float* const* weights, vsr_handle* out);

/* Re-pack after load_state_dict()/.to(): replaces nn.Module.load_state_dict coherence. */
int vsr_load_weights(vsr_handle h, const float* const* weights, void* stream);

void vsr_destroy(vsr_handle h);

/* Replaces the verb_2_vob_all JSON dict (controllable_captioning.py:25-34, 283-292) with a
 * CSR table: keys [host, n_keys, strictly increasing], offsets [host, n_keys+1],
 * vocab_idx [host, offsets[n_keys]].  n_keys = 0 clears the table. */
int vsr_set_verb_table(vsr_handle h, const int64_t* keys, const int32_t* offsets,
                       const int32_t* vocab_idx, int32_t n_keys);

/* Time-invariant part of step()/step_v() hoisted out of the loop
 * (controllable_captioning.py:126-128 / 203-205 image descriptor; :159/:240 validity of the
 * region rows; :161/:242 att_va projection of every slot tile; the img columns of
 * W1_is / lstm_cell_1.weight_ih / W1_ig (:151-152,181) and of lstm_cell_2.weight_ih (:174)).
 *   det       (b, D, F) fp32 (fp16 / bf16 through vsr_prologue_ex); det_batch_stride in elements, 0 when the caller expanded one
 *             image over all captions (eval_coco.py:243)
 *   det_seqs  (b, L, R, F) fp32 slot tiles, same dtype as det (feedback: statics[1]; teacher forcing: seqs[1], L=T)
 *   verbs     (b, L) or NULL; verbs_dtype one of VSR_DT_*; value -1 = no verb in that slot */
int vsr_prologue(vsr_handle h, const float* det, int64_t det_batch_stride, int32_t D,
                 const float* det_seqs, int32_t b, int32_t L, int32_t R,
                 const void* verbs, int32_t verbs_dtype, void* stream);

/* Index form of the prologue (SURVEY.md §8 f3; an ADDITIONAL fast entry point, not part of the reference's
 * call signature).  The reference's fields materialise every slot tile by copying detection rows
 * (data/field.py:461-541); here a slot is described by indices instead:
 *   slot_index (b, L, R) int32:  d >= 0  region = det[caption's image, d, :]
 *                                -2      region = mean of the image's valid detections (verb slots, field.py:460,517)
 *                                -1      padding
 * 10x fewer input bytes than det_seqs (b, L, R, F) and the att_va projection is computed once per detection row
 * instead of once per slot row.  Every decode entry point works unchanged after either prologue. */
int vsr_prologue_indexed(vsr_handle h, const float* det, int64_t det_batch_stride, int32_t D,
                         const int32_t* slot_index, int32_t b, int32_t L, int32_t R,
                         const void* verbs, int32_t verbs_dtype, void* stream);

/* Both prologues with the element type of the region features as an argument: feat_dtype is VSR_DT_F32, VSR_DT_F16
 * or VSR_DT_BF16 and applies to det and det_seqs alike (anything else is VSR_EINVAL).  det_batch_stride stays in
 * elements.  Feature pointers must be aligned to four elements (16 bytes in fp32, 8 bytes in half precision).
 * vsr_prologue / vsr_prologue_indexed are these calls with VSR_DT_F32.
 *   - Every kernel that reads features widens each value to fp32 as it loads it (exact) and then does the fp32
 *     arithmetic of the fp32 path in the same order, so a decode of half-precision features x is bit-identical to
 *     a decode of their fp32 upcast.  Only the bytes read change: half the copy and DRAM traffic of the features.
 *   - The index form's -2 rows (the image mean) stay fp32: the mean is computed in fp32 and never rounded.
 *   - The magnitude limit of the tensor-core operands (|feature| < 255 in the default f16+f8x2 mode) is unchanged;
 *     it bounds the activation scale, not the input format.
 *   - VSRDEC_GEMM=simt (the fp32 FFMA twin, a verification mode that reads det_seqs in place) takes fp32 features
 *     only: half precision returns VSR_EINVAL.
 * Every decode entry point works unchanged after either prologue, in any feature dtype. */
int vsr_prologue_ex(vsr_handle h, const void* det, int64_t det_batch_stride, int32_t D, const void* det_seqs,
                    int32_t b, int32_t L, int32_t R, int32_t feat_dtype, const void* verbs, int32_t verbs_dtype,
                    void* stream);
int vsr_prologue_indexed_ex(vsr_handle h, const void* det, int64_t det_batch_stride, int32_t D,
                            const int32_t* slot_index, int32_t b, int32_t L, int32_t R, int32_t feat_dtype,
                            const void* verbs, int32_t verbs_dtype, void* stream);

/* One decoder step for the b prologue captions, one row per caption
 * (ControllableCaptioningModel.step / step_v, controllable_captioning.py:117-190 / 192-297).
 *   h1,c1,h2,c2 (b,H) state in;  slot (b) int64 = slot index the row attends to (feedback:
 *   clamp(ctrl_det_idxs + prev_gate) as in :139-140; teacher forcing: t);  word (b) int64 input
 *   token (bos at t = 0, :136);  use_verbs/gt select step_v semantics.
 *   Outputs: h1o,c1o,h2o,c2o (b,H);  out_logp (b,V);  gate_logp (b,2). */
int vsr_step(vsr_handle h, const float* h1, const float* c1, const float* h2, const float* c2,
             const int64_t* slot, const int64_t* word, int32_t use_verbs, int32_t gt,
             float* h1o, float* c1o, float* h2o, float* c2o,
             float* out_logp, float* gate_logp, void* stream);

/* Whole beam search over the prologue batch without host synchronisation
 * (CaptioningModel.beam_search / beam_search_v, CaptioningModel.py:116-195 / 197-294).
 *   out_words,out_gates (b,out_size,T) int64;  lp_words,lp_gates (b,out_size,T) fp32
 *   eos_idxs[2] [host];  trace may be NULL.
 * Repeated calls with identical arguments (same prologue inputs, shapes and flags; trace == NULL) are replayed from a
 * CUDA graph that the library captures on an internal stream at the second such call and launches on `stream`
 * (vsr_prologue / vsr_prologue_indexed likewise).  If `stream` is itself being captured the work is enqueued as plain
 * launches.  VSRDEC_GRAPH=0 in the environment at vsr_create() time disables this. */
int vsr_beam_search(vsr_handle h, int32_t beam_size, int32_t out_size, const int64_t* eos_idxs,
                    int32_t use_verbs, int32_t gt,
                    int64_t* out_words, int64_t* out_gates, float* lp_words, float* lp_gates,
                    const VsrTrace* trace, void* stream);

/* Per-step selections of the last vsr_beam_search on this handle, each [T][b][beam]
 * (int32 parent slot / word / gate, fp32 accumulated score).  Any pointer may be NULL. */
int vsr_get_history(vsr_handle h, int32_t* parent, int32_t* word, int32_t* gate, float* score,
                    void* stream);

/* Teacher-forced unroll over the prologue batch (CaptioningModel.forward,
 * CaptioningModel.py:22-36; the prologue's det_seqs is seqs[1] with L = T).
 *   captions (b,T) int64;  out (b,T,V);  gate (b,T,2). */
int vsr_forward_teacher(vsr_handle h, const int64_t* captions, int32_t T,
                        float* out, float* gate, void* stream);

/* Greedy decode (CaptioningModel.test, CaptioningModel.py:38-52): argmax of both heads.
 *   out_words,out_gates (b,T) int64. */
int vsr_greedy(vsr_handle h, int64_t* out_words, int64_t* out_gates, void* stream);

/* Multinomial sampling decode with log-probs (CaptioningModel.sample_rl, CaptioningModel.py:54-76; caller
 * coco_scripts/train.py:151): at every step both heads are sampled from the step's distributions (word: Gumbel-max
 * over the vocabulary row with a Philox4x32-10 stream keyed by `seed`; gate: one uniform draw), the picks are fed
 * back, and the log-probs of the picks are returned.  The whole loop runs on the device.
 *   out_words,out_gates (b,T) int64;  lp_words,lp_gates (b,T) fp32.  The same seed reproduces the same draws.
 * Equal to vsr_sample_ex with {seed, 1, 1.f, 0, 1.f, 0, 0}. */
int vsr_sample(vsr_handle h, uint64_t seed, int64_t* out_words, int64_t* out_gates,
               float* lp_words, float* lp_gates, void* stream);

/* Sampling decode with several draws per caption, temperature, top-k / top-p truncation and verb forcing.
 * A call decodes the prologue's b captions with n >= 1 independent draws per caption.  Rows are caption-major:
 * row r = caption c = r / n, draw j = r % n.  Every row starts as init_state does; statics are read by c (no copy per
 * draw).  All T = seq_len steps run (no EOS stop).
 * At each step an UNFORCED row with vocabulary logits x (fp32), temperature tau, top_k and top_p:
 *   1. z_v = x_v / tau in fp32 (tau = 1 leaves x untouched).
 *   2. The vocabulary is ordered by (x desc, index asc): on x, not z, so that division rounding creates no new ties.
 *   3. Top-k: K = the first min(top_k, V) entries of that order; top_k = 0 means all V.
 *   4. Top-p: q_v = exp(z_v - max z) / sum_{u in K} exp(z_u - max z) over K; P = the shortest prefix of K, in the same
 *      order, whose mass is >= top_p.  top_p = 1 means P = K.  P always holds at least one word.
 *   5. word = argmax_{v in P} (z_v + G_v), ties by (value desc, index asc), G_v = -log(-log u_v) with u_v from the
 *      Philox4x32-10 counter (v >> 2, c, t, 2j), lane v & 3 (for j = 0 the numbers vsr_sample uses).  The gate is drawn
 *      from the step's gate log-probs with counter (0, c, t, 2j + 1); temperature and truncation apply to the word
 *      head only.
 *   6. lp_words = the MODEL's log-prob of the draw, (x_w - row max) - row log-sum-exp, unaffected by tau, top_k and
 *      top_p (what a scorer needs); lp_gates = the gate's log-prob, as vsr_sample returns them.
 * With use_verbs (vsr_step's use_verbs / gt semantics, gt as in vsr_beam_search; the prologue must have a verbs tensor)
 * a FORCED row (its current slot has a verb) takes the forced word with lp_word = 0 and gate 1 with lp_gate = 0.
 * Draw j of caption c is bit-identical for every n > j, and does not depend on b or on the other captions.  Masses
 * are summed in fixed point, so the top-p boundary does not depend on launch shape either.
 *   out_words,out_gates (b,n,T) int64;  lp_words,lp_gates (b,n,T) fp32.
 * z is clamped to +-FLT_MAX, so a tau small enough for x / tau to overflow float32 still gives a finite row: the
 * overflowing entries tie at FLT_MAX and are resolved in index order like any other tie.
 * VSR_EINVAL: n < 1, b * n > 2^30, tau not finite or <= 0, top_k < 0, top_p not in (0, 1], a null pointer, use_verbs
 * without a verbs tensor. */
typedef struct VsrSampleParams {
  uint64_t seed;
  int32_t n;            /* draws per caption, >= 1 */
  float temperature;    /* finite, > 0 */
  int32_t top_k;        /* >= 0, 0 = off */
  float top_p;          /* (0, 1], 1 = off */
  int32_t use_verbs;    /* step_v semantics: verb forcing (needs a prologue with verbs) */
  int32_t gt;
} VsrSampleParams;
int vsr_sample_ex(vsr_handle h, const VsrSampleParams* p, int64_t* out_words, int64_t* out_gates,
                  float* lp_words, float* lp_gates, void* stream);

/* Attention capture: where the decoder looks for every generated word.
 * vsr_set_attention_capture: while enabled, the decode drivers (vsr_beam_search, vsr_greedy, vsr_sample(_ex),
 *   vsr_forward_teacher) record, at every step and for every row, the R+1 attention weights of the slot attention
 *   (controllable_captioning.py:167-169) and the slot the row read, in a grow-only workspace of [T][rows][R+1] fp32 +
 *   [T][rows] int32 (8.4 MB at 1000 captions x beam 5 x R = 20).  Off by default; when off nothing is recorded and no
 *   launch or output changes.  Captured decodes replay from their own CUDA graphs.
 * vsr_get_attention: the attention of the last decode on the handle, enqueued on `stream` (no host synchronisation).
 *   vsr_beam_search:  alpha (b,out_size,T,R+1) fp32, slot (b,out_size,T) int32, following the back-pointer path of each
 *                     returned beam (the row whose distributions produced token t).  Note that lp_words / lp_gates are
 *                     NOT back-tracked (slot order, as in the reference), the attention is.
 *   vsr_sample_ex:    alpha (b,n,T,R+1), slot (b,n,T): draw j of caption c is row c*n + j.
 *   other drivers:    alpha (b,T,R+1), slot (b,T): one row per caption (T = the captions' length for teacher forcing).
 *   alpha[..., 0] is the sentinel weight and alpha[..., r+1] the weight of region r of the slot read at that step; the
 *   weights are exactly the ones that form the attended feature: 0 at padding regions and at an all-zero sentinel, the
 *   rest sums to 1.  Verb forcing does not change them.  After a caption's EOS the frozen beam keeps decoding and its
 *   weights are returned as computed, not masked.  R is the prologue's R at decode time.
 *   Returns VSR_ESTATE when the last decode ran without capture (or none has run). */
int vsr_set_attention_capture(vsr_handle h, int32_t enabled);
int vsr_get_attention(vsr_handle h, float* alpha, int32_t* slot, void* stream);

/* No-repeat n-gram blocking: a handle setting (like vsr_set_attention_capture) that applies to the decode drivers that
 * choose words, vsr_beam_search, vsr_greedy, vsr_sample and vsr_sample_ex (not vsr_step or vsr_forward_teacher).
 * n = 0 is off (the default): outputs, launches and graph replay are exactly those of a handle that never set it.
 * With block size n >= 1, a row's emitted words y_0 .. y_{t-1} are the words it picked at steps 0 .. t-1 (for beam
 * search the word path of the row's own beam, following the back-pointers; gates and BOS are not part of it).  At step
 * t, word w is BANNED for the row when some i with 0 <= i <= t - n has y_i .. y_{i+n-2} = y_{t-n+1} .. y_{t-1} and
 * y_{i+n-1} = w.  For n = 1 every word already emitted is banned.
 *   - A banned word cannot be selected.  Beam search: it is not among the row's word candidates (the top-k stays exact
 *     over the words that are not banned, ties in (value desc, index asc) order as always).  Greedy: the pick is the
 *     best word that is not banned.  Sampling (vsr_sample_ex): banned entries leave the row before steps 1-5, as if
 *     x_w = -inf, so K and P are taken over the words that are not banned.
 *   - Log-probs do not change: lp_words, the beam scores and the traced rows (VsrTrace.step_out) stay the model's own
 *     log-softmax over the full vocabulary, as the sampling log-probs ignore truncation.
 *   - A verb-forced row (use_verbs) takes the forced word even if it completes a banned n-gram; beams frozen by the
 *     double-EOS path (CaptioningModel.py:146-150) keep their synthetic candidates; blocking continues after a word EOS,
 *     since those beams keep expanding.
 *   - Each caption decodes to the same bits alone or with others, and sampling draw j is the same for every n > j.
 * Limits (VSR_EINVAL, nothing enqueued): 0 <= n <= seq_len here; with n >= 1, vsr_beam_search needs
 * vocab_size >= beam_size + seq_len - 1 and vsr_greedy / vsr_sample(_ex) need vocab_size >= seq_len, so that every row
 * keeps enough words that are not banned.  While on, the handle keeps a [rows][seq_len] int32 history of the decode's
 * words (two of them for beam search), allocated at the first decode that needs it. */
int vsr_set_no_repeat_ngram(vsr_handle h, int32_t n);

/* Diverse beam search (Vijayakumar et al., AAAI 2018): a handle setting (like vsr_set_no_repeat_ngram) that applies to
 * vsr_beam_search only (greedy, sampling, teacher forcing and vsr_step have no beams to group).  groups = 1 is off (the
 * default): outputs, launches and graph keys are exactly those of a handle that never set it, whatever the penalty.
 * With G = groups > 1, beam k, B = k / G beams per group and lambda = penalty, at step t for each caption:
 *   1. Group g owns beam slots [g*B, (g+1)*B) at every step.  At t = 0 every group expands the single BOS row (all 2k
 *      candidates); at t > 0 its candidates are the (parent j, word, gate) triples of its own slots j.  Candidate scores
 *      sc are the ones of the plain search: fl(seq + fl(word + gate)) for a live beam; for a beam frozen by the
 *      double-EOS path its old score at word 0 and -999 elsewhere.
 *   2. Groups choose in order g = 0, 1, ..., G-1.
 *   3. cnt_g(w) = the number of picks that groups 0 .. g-1 made AT THIS STEP whose word is w and whose parent is live
 *      (not frozen).  Picks of verb-forced rows count: they emit a real word.
 *   4. key = __fsub_rn(sc, __fmul_rn(lambda, (float)cnt_g(w))) for a candidate of a live row that is not verb-forced;
 *      key = sc otherwise (forced words and frozen beams' synthetic candidates are never penalised).
 *   5. Group g takes the B candidates with the largest key, ties by flat index ascending as always, in that order into
 *      its slots.  Two groups may take the same candidate at t = 0.
 *   6. The beam's accumulated score is sc, the model's own score, not key: the penalty steers the selection and is
 *      never accumulated.
 *   7. lp_words / lp_gates, the vsr_get_history scores and the traced rows (VsrTrace.step_out) stay the model's.
 *   8. The final ranking is the plain one: all k final beams sorted by score, the top out_size returned (out_size =
 *      beam_size returns every group's beams).
 * lambda = 0 with G > 1 is allowed: the groups are then independent searches of beam B (bit-identical to a plain
 * search of beam B except where two words of one row round to the same score: a group, which holds the row's top-k
 * words, then takes the lower word index by the tie rule).  A trace with forced selections
 * (VsrTrace.forced_*) replays them as always.  N-gram blocking composes (the candidates already exclude banned words);
 * attention capture is unchanged; each caption decodes to the same bits alone, stacked or sharded.
 * A penalty larger than the gap between a live score and -999 can rank a frozen beam's -999 synthetic candidates above
 * penalised live ones: the rule is still followed, those beams simply sort last.
 * Limits (VSR_EINVAL, nothing enqueued): 1 <= groups <= VSR_MAX_BEAM, penalty finite and >= 0; vsr_beam_search refuses
 * a beam_size that is not a multiple of groups. */
int vsr_set_beam_diversity(vsr_handle h, int32_t groups, float penalty);

/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t vsr_launch_count(vsr_handle h);

/* Which GEMM path this handle runs: "tcgen05-f16x3" (default: tcgen05.mma kind::f16 on fp16 hi/lo
 * splits, three MMAs per product into one fp32 TMEM accumulator) or "simt-fp32" (FFMA verification
 * twin, selected with VSRDEC_GEMM=simt at create time). */
const char* vsr_gemm_kind(vsr_handle h);

/* Per-phase device time of the last decode when enabled (CUDA events around each phase of each
 * step; adds event overhead, off by default).  names/ms are [host] arrays of capacity cap;
 * returns the number of phases written, or a negative error. */
int vsr_set_profiling(vsr_handle h, int32_t enabled);
int vsr_get_phase_times(vsr_handle h, const char** names, float* ms, int32_t* launches, int32_t cap);
/* Device time of every decoder step (decoder step + beam selection/reorder) of the last vsr_beam_search run with
 * profiling enabled: CUDA events between the steps on the launching stream (SURVEY.md 8d "p50 per-step latency").
 * ms is a [host] array of capacity cap; returns the number of steps written, or a negative error. */
int vsr_get_step_times(vsr_handle h, float* ms, int32_t cap);

/* ------------------------------------------------------------------------------------------------------------------
 * R-level SSP of the eval pre-step (SURVEY.md 8 f2): SinkhornNet forward + optimal assignment, batched.
 * Replaces models/sinkhorn_network.py:30-51 (SinkhornNet.forward / sinkhorn) and the per-role
 * `.cpu()` + `munkres.Munkres().compute(make_cost_matrix(mx))` of coco_scripts/eval_coco.py:184-189 (flickr_scripts/
 * eval_flickr.py likewise).  `weights` [host array of 10 device pointers] follows the state_dict order:
 *   W1_txt.weight (128,300) .bias | W1_vis.weight (512,2048) .bias | W2_vis.weight (128,512) .bias |
 *   W_fc_pos.weight (256,260) .bias | W_fc.weight (N,256) .bias          (sinkhorn_network.py:11-15)
 * vsr_ssp_create:  N in [1,16], and only if the whole network of one problem fits a block's opt-in shared memory on the
 *   current device (218,368 B at N = 16; 227 KB on a B200): every N it accepts runs at every batch size.
 * vsr_ssp_forward:  seq (B,N,2352) fp32 rows, split by column as sinkhorn_network.py:39-41 slices them: [0,300) -> W1_txt,
 *   [300,2348) -> W1_vis, [2348,2352) appended before W_fc_pos (the eval feeds the concatenation of eval_coco.py:146 unchanged);
 *   matrix (B,N,N) fp32 = SinkhornNet(seq);  assign (B,N) int32 or NULL = for every row r of matrix^T (the profit matrix
 *   of eval_coco.py:187) the column of its maximum-profit assignment (what munkres returns as pairs (r, col)). */
typedef struct VsrSspHandle_* vsr_ssp_handle;
int vsr_ssp_create(const float* const* weights, int32_t N, int32_t n_iters, float tau, vsr_ssp_handle* out);
int vsr_ssp_load_weights(vsr_ssp_handle h, const float* const* weights, void* stream);
void vsr_ssp_destroy(vsr_ssp_handle h);
int vsr_ssp_forward(vsr_ssp_handle h, const float* seq, int32_t B, float* matrix, int32_t* assign, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * S-level SSP of the eval pre-step (SURVEY.md 8 f2): the semantic-role sorter, batched.
 * Replaces models/sort_model.py:105-119, 149-183 (S_SSP.generate(mode='not-normal')) with its encoder / decoder stacks
 * (models/sort_modules.py:52-63, 79-99, 120-135; models/transformer_modules.py:36-54, 104-134, 188-212, 325-346) as
 * coco_scripts/eval_coco.py:170-174 calls them once per (caption, verb) with batch 1.
 * `weights` [host array of n_weights = 10 + 34 * n_layers device pointers], in this order (state_dict names):
 *   sr_embed_layer.weight (n_roles,d) | v_embed_layer.weight (n_verbs,d) | encoder.fc_feat.weight (d,d) .bias (both NULL when
 *   add_fc = 0) | encoder.layer_norm.weight .bias |
 *   per encoder layer l: attention.linear_{Q,K,V,O}.{weight,bias} | ff_layer.w_1.{weight,bias} | ff_layer.w_2.{weight,bias} |
 *                        layer_norm1.{weight,bias} | layer_norm2.{weight,bias}                                    (16 pointers)
 *   decoder.layer_norm.weight .bias |
 *   per decoder layer l: attention.linear_{Q,K,V,O}.{weight,bias} | ff_layer.w_1 | ff_layer.w_2 | layer_norm1..3  (18 pointers;
 *                        the checkpoint's cross_attention.* tensors are never used by the reference, sort_modules.py:88)
 *   expander_nn.weight (n_roles,d) .bias
 * vsr_sort_generate: P independent problems.  verbs (P) int64 (already taken modulo 10000, sort_model.py:108), roles (P,max_len)
 *   int64 = the problem's distinct non-zero role ids, zero padded (ids outside [0,n_roles) / [0,n_verbs) are clamped);
 *   n_steps decoder steps are run (the largest role count of the batch is enough; <= max_len);  pred (P,max_len) int64 = role
 *   ids in generated order, logp (P,max_len) fp32 = log-prob of each choice, both zero after a problem's last role;
 *   step_rows (P,n_steps,n_roles) fp32 or NULL = the log-softmax row of every step.  n_active [host, n_steps] or NULL: when the
 *   caller has sorted the problems by falling role count, n_active[t] = number of problems with more than t roles — the
 *   decoder steps then run on the first n_active[t] problems only.  No host synchronisation. */
typedef struct VsrSortDims {
  int32_t n_roles;   /* 26 */
  int32_t n_verbs;   /* rows of v_embed_layer: 2663 (coco) / 2927 (flickr) */
  int32_t d_model;   /* 512 */
  int32_t d_ff;      /* 2048 */
  int32_t n_heads;   /* 8 */
  int32_t n_layers;  /* 3 encoder + 3 decoder layers */
  int32_t max_len;   /* 10 */
  int32_t add_fc;    /* encoder.fc_feat present */
} VsrSortDims;
typedef struct VsrSortHandle_* vsr_sort_handle;
int vsr_sort_create(const VsrSortDims* dims, const float* const* weights, int32_t n_weights, vsr_sort_handle* out);
int vsr_sort_load_weights(vsr_sort_handle h, const float* const* weights, int32_t n_weights, void* stream);
void vsr_sort_destroy(vsr_sort_handle h);
int vsr_sort_generate(vsr_sort_handle h, const int64_t* verbs, const int64_t* roles, int32_t P, int32_t n_steps,
                      const int32_t* n_active, int64_t* pred, float* logp, float* step_rows, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Host bookkeeping of the eval pre-step (SURVEY.md 8 f2), for a whole batch of captions: the integer logic of
 * coco_scripts/eval_coco.py:148-237 around the two device networks.  HOST pointers throughout; no CUDA call inside.
 * vsr_preorder_begin: control_verb (C,n_verb), det_seqs_v / det_seqs_sr (C,L,n_verb) int64 -> the (caption, verb) problems
 *   (eval_coco.py:148-171: distinct roles in first-seen order, at most `limit`; the slots holding each; roles held by several
 *   slots); N = sinkhorn_len, fixed_len = slots per caption.  Returns the number of S-level problems, of R-level problems
 *   (repeated roles) and the largest role count.
 * vsr_preorder_fill: inputs of the two batched device calls — verbs (P), roles (P,roles_ld) zero padded, counts (P), and for
 *   every repeated role the rows of its slots in the (C*fixed_len, 2352) row matrix: gather (n_repeated,N), -1 = zero row
 *   (eval_coco.py:176-182).  Any output may be NULL.
 * vsr_preorder_end: pred (P,pred_ld) = vsr_sort_generate's orders, assign (n_repeated,N) = vsr_ssp_forward's assignments,
 *   slot_valid (C,fixed_len) u8 = slots whose tile is not empty (:226), verb_list (C,fixed_len) f64 -> src_slot (C,fixed_len)
 *   int64 (row j of the re-ordered caption is slot src_slot[c][j]; empty tiles dropped, tail repeating the last kept slot,
 *   :217-231) and verbs_out (C,fixed_len) f32 (:234-235); region order (:190-200), rank assembly (:202-209) and
 *   verb_rank_merge (utils/tools.py:35-71) happen here.  Frees the handle (vsr_preorder_free: for an abandoned one). */
typedef struct VsrPreorderHandle_* vsr_preorder_handle;
int vsr_preorder_begin(const int64_t* control_verb, const int64_t* det_seqs_v, const int64_t* det_seqs_sr, int32_t C,
                       int32_t n_verb, int32_t L, int32_t limit, int32_t N, int32_t fixed_len, vsr_preorder_handle* out,
                       int32_t* n_problems, int32_t* n_repeated, int32_t* max_roles);
int vsr_preorder_fill(vsr_preorder_handle h, int64_t* verbs, int64_t* roles, int32_t roles_ld, int32_t* counts, int64_t* gather);
int vsr_preorder_end(vsr_preorder_handle h, const int64_t* pred, int32_t pred_ld, const int32_t* assign,
                     const uint8_t* slot_valid, const double* verb_list, int64_t* src_slot, float* verbs_out);
void vsr_preorder_free(vsr_preorder_handle h);

#ifdef __cplusplus
}
#endif
#endif /* VSRDEC_H_ */
