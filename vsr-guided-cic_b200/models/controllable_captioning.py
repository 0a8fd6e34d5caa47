"""Role-shift captioning decoder, B200-native drop-in.

Keeps the reference's class surface (models/controllable_captioning.py:10-303): constructor
signature, the 28-tensor state_dict (same names, shapes, dtypes, registration order),
`init_state`, `step`, `step_v`, `test`, `sample_rl`, and the inherited `forward` /
`beam_search` / `beam_search_v`.  `sample_rl` and the inherited `sample_v` (sampling with verb forcing) also take
n draws per caption, a temperature and top-k / top-p truncation (models/CaptioningModel.py).  Every decode driver also returns the per-word attention on request
(`return_attention=True`, see models/CaptioningModel.py), which the reference only exposes as a local of `step_v`.
Region features (detections, det_seqs / ctrl_det_seqs) may be float16 or bfloat16 as well as float32: a decode of
half-precision features is bit-identical to the decode of their float32 upcast, and reads half the bytes.  The parameters live in ordinary torch modules so that
`.to()`, `.eval()`, `load_state_dict()` work unchanged; all arithmetic of the hot path runs in
libvsrdec's sm_100a kernels on a packed copy of the weights that is rebuilt whenever the
parameters change.  CPU tensors raise: this path has no fallback.

LIMITS the reference does not have (each raises VsrError with a message, never a silent wrong result):
  * CUDA tensors only; parameters and inputs on one device;
  * beam_size <= 8 (VSR_MAX_BEAM: the fused per-caption selection keeps 2*beam^2 candidates in one warp);
  * <= 64 regions per slot (the slot validity mask is one 64-bit word);
  * det_feat_size % 4 == 0 and att_size % 4 == 0 (128-bit loads); vocab_size <= 49152; vocab_size >= beam_size;
  * seq_len <= 256 for beam search (back-track kernel's shared-memory history);
  * tensor-core operands are carried as fp16 (+ fp16 / e4m3 residuals): weights are rescaled per tensor by a power of
    two, activations are not — hidden states are in [-1, 1] by construction, region features must stay below 255 in
    magnitude in the default "f16+f8x2" GEMM mode (65504 with VSRDEC_GEMM=f16x3); larger values saturate.  The bound is
    on the activation scale, not the input format: it is the same for float32, float16 and bfloat16 features;
  * region features are float32, float16 or bfloat16, one dtype for the detections and the slot tiles (a mismatch or
    any other dtype raises); half precision is refused under VSRDEC_GEMM=simt (the fp32 FFMA verification twin).
  * sampling (`sample_rl`, `sample_v`): captions x n draws <= 2^30 rows per call; temperature a finite float32 > 0 and
    top_p in (0, 1] as float32 values (where logits / temperature overflows float32 it is clamped to +-FLT_MAX: the
    overflowing words tie and the lowest index among them wins).
Among candidates whose fp32 scores tie EXACTLY the order is (score desc, flat index asc); torch.sort leaves it unspecified.
"""
import json
import os

import torch
from torch import nn

from .CaptioningModel import CaptioningModel as _CaptioningModel

_TABLE_FILES = {  # CWD-relative, as in the reference (controllable_captioning.py:25-34)
    'coco': ('datasets/coco', 'verb_2_vob_all_refine.json', 'verb_2_vob.json'),
    'flickr': ('datasets/flickr', 'verb_2_vob_all_refine_flickr.json', 'verb_2_vob_flickr.json'),
}


class ControllableCaptioningModel(_CaptioningModel):
    def __init__(self, seq_len, vocab_size, bos_idx, det_feat_size=2048, input_encoding_size=1000,
                 rnn_size=1000, att_size=512, h2_first_lstm=True, img_second_lstm=False, dataset='coco',
                 *, verb_tables=None):
        super().__init__(seq_len)
        self.vocab_size = vocab_size
        self.bos_idx = bos_idx
        self.det_feat_size = det_feat_size
        self.input_encoding_size = input_encoding_size
        self.rnn_size = rnn_size
        self.att_size = att_size
        self.h2_first_lstm = h2_first_lstm
        self.img_second_lstm = img_second_lstm

        if verb_tables is not None:       # extension: pass the two dicts instead of reading the JSON files
            self.verb_2_vob_all, self.verb_2_vob = verb_tables
        else:
            folder, f_all, f_one = _TABLE_FILES['coco' if dataset == 'coco' else 'flickr']
            with open(os.path.join(folder, f_all)) as f:
                self.verb_2_vob_all = json.load(f)
            with open(os.path.join(folder, f_one)) as f:
                self.verb_2_vob = json.load(f)

        H, E, Fd, A = rnn_size, input_encoding_size, det_feat_size, att_size
        in1 = Fd + E + (H if h2_first_lstm else 0)        # input_1 = [h2 | img | xt]
        in2 = H + Fd + (Fd if img_second_lstm else 0)     # input_2 = [h1 | att | img]
        # registration order defines the state_dict order (and the C ABI's weight order)
        self.embed = nn.Embedding(vocab_size, E)
        self.W1_is = nn.Linear(in1, H)
        self.W1_hs = nn.Linear(H, H)
        self.att_va = nn.Linear(Fd, A, bias=False)
        self.att_ha = nn.Linear(H, A, bias=False)
        self.att_a = nn.Linear(A, 1, bias=False)
        self.att_sa = nn.Linear(H, A, bias=False)
        self.att_s = nn.Linear(A, 1, bias=False)
        self.lstm_cell_1 = nn.LSTMCell(in1, H)
        self.lstm_cell_2 = nn.LSTMCell(in2, H)
        self.out_fc = nn.Linear(H, vocab_size)
        self.s_fc = nn.Linear(H, Fd)
        self.W1_ig = nn.Linear(in1, H)
        self.W1_hg = nn.Linear(H, H)
        self.att_ga = nn.Linear(H, A, bias=False)
        self.att_g = nn.Linear(A, 1, bias=False)

        self._eng = None
        self._eng_key = None
        self._table_key = None
        self._prologue_key = None
        self._prologue_refs = None
        self.init_weights()

    # ------------------------------------------------------------------ parameters
    def init_weights(self):
        """Same initialisers, in the same order, as the reference (controllable_captioning.py:72-107):
        Xavier-normal matrices, orthogonal LSTM recurrences, zero biases."""
        xavier = [self.embed.weight, self.out_fc.weight, self.s_fc.weight, self.W1_is.weight,
                  self.W1_hs.weight, self.att_va.weight, self.att_ha.weight, self.att_a.weight,
                  self.att_sa.weight, self.att_s.weight]
        for w in xavier:
            nn.init.xavier_normal_(w)
        for cell in (self.lstm_cell_1, self.lstm_cell_2):
            nn.init.xavier_normal_(cell.weight_ih)
            nn.init.orthogonal_(cell.weight_hh)
        for w in (self.W1_ig.weight, self.W1_hg.weight, self.att_ga.weight, self.att_g.weight):
            nn.init.xavier_normal_(w)
        for name, p in self.named_parameters():
            if 'bias' in name:
                nn.init.constant_(p, 0)

    def init_state(self, b_s, device):
        """(reference controllable_captioning.py:109-115)"""
        z = lambda: torch.zeros((b_s, self.rnn_size), device=device)
        return (z(), z()), (z(), z()), torch.zeros((b_s,), dtype=torch.long, device=device)

    def _dims(self):
        return dict(seq_len=self.seq_len, vocab_size=self.vocab_size, bos_idx=self.bos_idx,
                    det_feat_size=self.det_feat_size, input_encoding_size=self.input_encoding_size,
                    rnn_size=self.rnn_size, att_size=self.att_size,
                    h2_first_lstm=int(bool(self.h2_first_lstm)), img_second_lstm=int(bool(self.img_second_lstm)))

    def _engine(self):
        """The per-device libvsrdec handle, (re)packed when parameters moved or changed."""
        from vsrdec import DecoderEngine, PARAM_NAMES, VsrError
        sd = dict(self.named_parameters())
        ws = [sd[n] for n in PARAM_NAMES]
        if not ws[0].is_cuda:
            raise VsrError("ControllableCaptioningModel: parameters are on the CPU; this decoder path "
                           "runs only on a CUDA device (no CPU fallback) — call .to('cuda') first")
        key = tuple((w.data_ptr(), w._version, w.device) for w in ws)
        if self._eng is None or self._eng.device != ws[0].device:
            if self._eng is not None:
                self._eng.close()
            self._eng = DecoderEngine(self._dims(), ws)
            self._table_key = None
            self._prologue_key = None
        elif key != self._eng_key:
            self._eng.load_weights(ws)
            self._prologue_key = None
        self._eng_key = key
        tkey = id(self.verb_2_vob_all), len(self.verb_2_vob_all)
        if tkey != self._table_key:
            self._eng.set_verb_table(self.verb_2_vob_all)
            self._table_key = tkey
        return self._eng

    @staticmethod
    def _tkey(t):
        return None if t is None else (t.data_ptr(), t._version, tuple(t.shape), tuple(t.stride()), t.dtype)

    def _engine_for(self, statics, seqs=None, reuse=False):
        """Engine with the prologue (time-invariant terms) computed for these statics.  The decode
        drivers always recompute it; the single-step API (`reuse=True`) skips it while it is handed
        the very same (unmodified) tensors, which are kept referenced so their storage cannot be
        recycled under the cache key."""
        eng = self._engine()
        det = statics[0]
        if seqs is not None:                  # teacher forcing: slot tiles come from seqs[1] (:131-133)
            det_seqs, verbs = seqs[1], None
        else:
            det_seqs = statics[1]
            verbs = statics[2] if len(statics) > 2 else None
        key = (self._tkey(det), self._tkey(det_seqs), self._tkey(verbs))
        if not reuse or key != self._prologue_key:
            eng.prologue(det, det_seqs, verbs)
            self._prologue_key = key
            self._prologue_refs = (det, det_seqs, verbs)
        return eng

    # ------------------------------------------------------------------ single steps
    def _step_impl(self, t, state, prev_outputs, statics, seqs, mode, use_verbs, gt):
        assert (mode in ['teacher_forcing', 'feedback'])
        (h1, c1), (h2, c2), ctrl_det_idxs = state
        b_s = statics[0].size(0)
        device = statics[0].device
        if mode == 'teacher_forcing':
            if use_verbs:   # the reference's step_v reads verb_curr, which only feedback mode defines
                raise NameError("step_v supports mode='feedback' only")
            eng = self._engine_for(statics, seqs, reuse=True)
            word = seqs[0][:, t]
            slot = torch.full((b_s,), t, dtype=torch.long, device=device)
        else:
            eng = self._engine_for(statics, reuse=True)
            if t == 0:
                word = torch.full((b_s,), self.bos_idx, dtype=torch.long, device=device)
            else:
                word = prev_outputs[0]
                ctrl_det_idxs = torch.clamp(ctrl_det_idxs + prev_outputs[1], 0, statics[1].shape[1] - 1)
            slot = ctrl_det_idxs
        (out, gate), (h1n, c1n, h2n, c2n) = eng.step(h1, c1, h2, c2, slot, word, use_verbs=use_verbs, gt=gt)
        return (out, gate), ((h1n, c1n), (h2n, c2n), ctrl_det_idxs)

    def step(self, t, state, prev_outputs, statics, seqs, *args, mode='teacher_forcing'):
        ''' statics[0]: (b_s, det_len, feat_dim), statics[1]: (b_s, fixed_len, max_det, feat_dim)
            (reference controllable_captioning.py:117-190) '''
        return self._step_impl(t, state, prev_outputs, statics, seqs, mode, False, False)

    def step_v(self, t, state, prev_outputs, statics, seqs, *args, mode='teacher_forcing', gt=False):
        ''' as step, plus statics[2]: (b_s, fixed_len) verb ids, -1 = none
            (reference controllable_captioning.py:192-297) '''
        return self._step_impl(t, state, prev_outputs, statics, seqs, mode, True, gt)

    def test(self, detections, ctrl_det_seqs_test, return_attention=False):
        return super().test((detections, ctrl_det_seqs_test), return_attention=return_attention)

    def sample_rl(self, detections, ctrl_det_seqs_test, seed=None, return_attention=False, n=1, temperature=1.0,
                  top_k=0, top_p=1.0):
        return super().sample_rl((detections, ctrl_det_seqs_test), seed=seed, return_attention=return_attention, n=n,
                                 temperature=temperature, top_k=top_k, top_p=top_p)
