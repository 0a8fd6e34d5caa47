"""DecoderEngine: thin, torch-aware wrapper over the C ABI (one handle per device).

PyTorch is plumbing here (device memory, streams); every hot operation runs in libvsrdec's
sm_100a kernels.  CPU tensors are rejected — there is no fallback path."""
import ctypes
import math
import numbers
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib
from ._lib import VsrError, VsrDims, VsrSampleParams, VsrTrace, c_vp, c_i32, c_i64, c_f

# state_dict registration order of the reference model (controllable_captioning.py:23-68);
# the order of the `weights` array of vsr_create().
PARAM_NAMES = (
    "embed.weight", "W1_is.weight", "W1_is.bias", "W1_hs.weight", "W1_hs.bias", "att_va.weight",
    "att_ha.weight", "att_a.weight", "att_sa.weight", "att_s.weight",
    "lstm_cell_1.weight_ih", "lstm_cell_1.weight_hh", "lstm_cell_1.bias_ih", "lstm_cell_1.bias_hh",
    "lstm_cell_2.weight_ih", "lstm_cell_2.weight_hh", "lstm_cell_2.bias_ih", "lstm_cell_2.bias_hh",
    "out_fc.weight", "out_fc.bias", "s_fc.weight", "s_fc.bias", "W1_ig.weight", "W1_ig.bias",
    "W1_hg.weight", "W1_hg.bias", "att_ga.weight", "att_g.weight")

_VERB_DT = {torch.float64: 0, torch.float32: 1, torch.int64: 2}
# element types of the region features (VSR_DT_F32 / F16 / BF16): a half-precision decode is bit-identical to the
# decode of its fp32 upcast (the kernels widen every value as they load it)
_FEAT_DT = {torch.float32: 1, torch.float16: 3, torch.bfloat16: 4}


def _stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _feat_dtype(*feats):
    """dtype tag of the feature tensors, which must share one of float32 / float16 / bfloat16."""
    dt = feats[0][0].dtype
    for t, name in feats:
        if t.dtype not in _FEAT_DT:
            raise VsrError(f"{name} must be torch.float32, torch.float16 or torch.bfloat16, got {t.dtype}")
        if t.dtype != dt:
            raise VsrError(f"detections and det_seqs must share one dtype, got {dt} and {t.dtype}")
    return _FEAT_DT[dt]


MAX_SAMPLE_ROWS = 2 ** 30       # captions x draws of one sampling call (vsr_sample_ex)


def check_sample_args(n, temperature, top_k, top_p, b=None):
    """Raise VsrError unless (n, temperature, top_k, top_p) are valid sampling parameters (vsr_sample_ex) for b
    captions.  temperature and top_p are checked as the float32 values the library receives: a finite temperature that
    rounds to 0 in float32 (e.g. 1e-50) is refused here, not after the prologue has run."""
    if isinstance(n, bool) or not isinstance(n, numbers.Integral) or not 1 <= n < 2 ** 31:
        raise VsrError(f"n (draws per caption) must be an int >= 1, got {n!r}")
    if b is not None and b * n > MAX_SAMPLE_ROWS:
        raise VsrError(f"{b} captions x n={n} draws exceed {MAX_SAMPLE_ROWS} rows per sampling call")
    if isinstance(top_k, bool) or not isinstance(top_k, numbers.Integral) or top_k < 0:
        raise VsrError(f"top_k must be an int >= 0 (0 = off), got {top_k!r}")
    try:
        tau, p = float(temperature), float(top_p)
    except (TypeError, ValueError):
        raise VsrError(f"temperature and top_p must be numbers, got {temperature!r} / {top_p!r}") from None
    tau32, p32 = c_f(tau).value, c_f(p).value
    if not math.isfinite(tau32) or tau32 <= 0.0:
        raise VsrError(f"temperature must be a finite float32 > 0, got {temperature!r}")
    if not (0.0 < p <= 1.0) or p32 <= 0.0:
        raise VsrError(f"top_p must be in (0, 1] (1 = off) and nonzero in float32, got {top_p!r}")


def check_no_repeat_ngram(n, seq_len, vocab_size=None, beam_size=1):
    """Raise VsrError unless n is a valid no-repeat n-gram block size (vsr_set_no_repeat_ngram) for a model of seq_len
    steps: an int in [0, seq_len].  With vocab_size, also for a decode with beam_size rows per caption (1: greedy and
    sampling): when on, vocab_size >= beam_size + seq_len - 1, so that every row keeps enough words that are not banned."""
    if isinstance(n, bool) or not isinstance(n, numbers.Integral) or not 0 <= n <= seq_len:
        raise VsrError(f"no_repeat_ngram_size must be an int in [0, seq_len={seq_len}] (0 = off), got {n!r}")
    if n > 0 and vocab_size is not None and vocab_size < beam_size + seq_len - 1:
        raise VsrError(f"no_repeat_ngram_size={n} needs vocab_size >= beam + seq_len - 1 = {beam_size + seq_len - 1}, "
                       f"got {vocab_size}")


MAX_BEAM = 8                    # VSR_MAX_BEAM


def check_beam_diversity(groups, penalty, beam_size=None):
    """Raise VsrError unless (groups, penalty) is a valid diverse beam search setting (vsr_set_beam_diversity): groups an
    int in [1, 8] (1 = off), penalty a real number, finite and >= 0 as a float32.  With beam_size, also for a beam search
    of that size: beam_size must be a multiple of groups."""
    if isinstance(groups, bool) or not isinstance(groups, numbers.Integral) or not 1 <= groups <= MAX_BEAM:
        raise VsrError(f"num_beam_groups must be an int in [1, {MAX_BEAM}] (1 = off), got {groups!r}")
    if isinstance(penalty, bool) or not isinstance(penalty, numbers.Real):
        raise VsrError(f"diversity_penalty must be a real number >= 0, got {penalty!r}")
    p32 = c_f(float(penalty)).value
    if not math.isfinite(p32) or not p32 >= 0.0:
        raise VsrError(f"diversity_penalty must be finite and >= 0 in float32, got {penalty!r}")
    if beam_size is not None and beam_size % groups != 0:
        raise VsrError(f"beam_size={beam_size} is not a multiple of num_beam_groups={groups}")


def _req_cuda(t: torch.Tensor, name: str, dtype=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise VsrError(f"{name} must be a CUDA tensor (no CPU fallback on this path)")
    if dtype is not None and t.dtype != dtype:
        raise VsrError(f"{name} must be {dtype}, got {t.dtype}")
    return t


class DecoderEngine:
    def __init__(self, dims: Dict, weights: Sequence[torch.Tensor]):
        self.lib = _lib.load_library()
        self.dims = dict(dims)
        self.device = weights[0].device
        self._keep = None
        self._weights = None
        self._attn_shape = None
        self.no_repeat_ngram = 0
        self.beam_diversity = (1, 0.0)
        self.handle = c_vp()
        d = VsrDims(*(int(self.dims[k]) for k in ("seq_len", "vocab_size", "bos_idx", "det_feat_size",
                                                   "input_encoding_size", "rnn_size", "att_size",
                                                   "h2_first_lstm", "img_second_lstm")))
        arr = self._weight_array(weights)
        with torch.cuda.device(self.device):
            torch.cuda.current_stream(self.device).synchronize()
            _lib.check(self.lib, self.lib.vsr_create(ctypes.byref(d), arr, ctypes.byref(self.handle)))

    def _weight_array(self, weights):
        if len(weights) != len(PARAM_NAMES):
            raise VsrError(f"expected {len(PARAM_NAMES)} weight tensors, got {len(weights)}")
        ws = []
        for name, w in zip(PARAM_NAMES, weights):
            _req_cuda(w, name, torch.float32)
            if w.device != self.device:
                raise VsrError("all parameters must live on one device")
            ws.append(w.detach().contiguous())
        self._weights = ws      # keep the (possibly re-laid-out) tensors alive during packing
        return (c_vp * len(ws))(*[w.data_ptr() for w in ws])

    def load_weights(self, weights):
        arr = self._weight_array(weights)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_load_weights(self.handle, arr, _stream_ptr(self.device)))

    def close(self):
        if getattr(self, "handle", None) is not None and self.handle.value:
            self.lib.vsr_destroy(self.handle)
            self.handle = c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ verb table
    def set_verb_table(self, table: Optional[Dict[str, List[int]]]):
        """`table` has the JSON shape of verb_2_vob_all: {str(verb_id): [vocab idx, ...]}."""
        items = []
        for k, v in (table or {}).items():
            try:
                key = int(k)
            except ValueError:
                continue   # str(int) keys only can ever match str(verb_curr.item())
            if str(key) != k:
                continue
            items.append((key, [int(x) for x in v]))
        items.sort()
        n = len(items)
        keys = (c_i64 * max(n, 1))(*[k for k, _ in items])
        offs = [0]
        flat = []
        for _, v in items:
            flat.extend(v)
            offs.append(len(flat))
        offsets = (c_i32 * (n + 1))(*offs)
        idx = (c_i32 * max(len(flat), 1))(*flat)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_set_verb_table(self.handle, keys, offsets, idx, n))

    # ------------------------------------------------------------------ prologue
    def prologue(self, det: torch.Tensor, det_seqs: torch.Tensor, verbs: Optional[torch.Tensor] = None):
        """det (b, D, F) and det_seqs (b, L, R, F) in one of float32 / float16 / bfloat16."""
        _req_cuda(det, "detections")
        _req_cuda(det_seqs, "det_seqs")
        fdt = _feat_dtype((det, "detections"), (det_seqs, "det_seqs"))
        if det.dim() != 3 or det_seqs.dim() != 4 or det.size(0) != det_seqs.size(0):
            raise VsrError(f"bad static shapes {tuple(det.shape)} / {tuple(det_seqs.shape)}")
        F = self.dims["det_feat_size"]
        if det.size(2) != F or det_seqs.size(3) != F:
            raise VsrError("feature width does not match det_feat_size")
        b, D = det.size(0), det.size(1)
        if b > 1 and det.stride(0) == 0 and det[0].is_contiguous():
            det_k, stride = det[0], 0           # one image expanded over all captions (eval_coco.py:243)
        else:
            det_k = det.contiguous()
            stride = D * F
        ds = det_seqs.contiguous()
        vb, vdt = None, 0
        if verbs is not None:
            _req_cuda(verbs, "verbs")
            if verbs.dtype not in _VERB_DT:
                verbs = verbs.double()
            if tuple(verbs.shape) != (b, ds.size(1)):
                raise VsrError(f"verbs shape {tuple(verbs.shape)} != {(b, ds.size(1))}")
            vb = verbs.contiguous()
            vdt = _VERB_DT[vb.dtype]
        self._keep = (det_k, ds, vb)
        self.b, self.L, self.R = b, ds.size(1), ds.size(2)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_prologue_ex(
                self.handle, det_k.data_ptr(), stride, D, ds.data_ptr(), b, self.L, self.R, fdt,
                vb.data_ptr() if vb is not None else None, vdt, _stream_ptr(self.device)))

    def prologue_indexed(self, det: torch.Tensor, slot_index: torch.Tensor, verbs: Optional[torch.Tensor] = None):
        """Index form of the prologue (vsr_prologue_indexed): slot_index (b, L, R) holds, per region, a
        detection row of the caption's image (>= 0), -2 for the image's mean row, or -1 for padding.  det is
        float32, float16 or bfloat16; the mean rows are computed and read in fp32 whatever its dtype."""
        _req_cuda(det, "detections")
        fdt = _feat_dtype((det, "detections"))
        _req_cuda(slot_index, "slot_index")
        if det.dim() != 3 or slot_index.dim() != 3 or det.size(0) != slot_index.size(0):
            raise VsrError(f"bad static shapes {tuple(det.shape)} / {tuple(slot_index.shape)}")
        F = self.dims["det_feat_size"]
        if det.size(2) != F:
            raise VsrError("feature width does not match det_feat_size")
        b, D = det.size(0), det.size(1)
        if b > 1 and det.stride(0) == 0 and det[0].is_contiguous():
            det_k, stride = det[0], 0
        else:
            det_k = det.contiguous()
            stride = D * F
        idx = slot_index.to(torch.int32).contiguous()
        vb, vdt = None, 0
        if verbs is not None:
            _req_cuda(verbs, "verbs")
            if verbs.dtype not in _VERB_DT:
                verbs = verbs.double()
            if tuple(verbs.shape) != (b, idx.size(1)):
                raise VsrError(f"verbs shape {tuple(verbs.shape)} != {(b, idx.size(1))}")
            vb = verbs.contiguous()
            vdt = _VERB_DT[vb.dtype]
        self._keep = (det_k, idx, vb)
        self.b, self.L, self.R = b, idx.size(1), idx.size(2)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_prologue_indexed_ex(
                self.handle, det_k.data_ptr(), stride, D, idx.data_ptr(), b, self.L, self.R, fdt,
                vb.data_ptr() if vb is not None else None, vdt, _stream_ptr(self.device)))

    # ------------------------------------------------------------------ single step
    def step(self, h1, c1, h2, c2, slot, word, use_verbs=False, gt=False):
        b, H, V = self.b, self.dims["rnn_size"], self.dims["vocab_size"]
        st = [_req_cuda(x, "state", torch.float32).contiguous() for x in (h1, c1, h2, c2)]
        for x in st:
            if tuple(x.shape) != (b, H):
                raise VsrError(f"state shape {tuple(x.shape)} != {(b, H)}")
        slot = _req_cuda(slot, "slot").long().contiguous()
        word = _req_cuda(word, "word").long().contiguous()
        new = [torch.empty((b, H), device=self.device, dtype=torch.float32) for _ in range(4)]
        out = torch.empty((b, V), device=self.device, dtype=torch.float32)
        gate = torch.empty((b, 2), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_step(
                self.handle, *[x.data_ptr() for x in st], slot.data_ptr(), word.data_ptr(),
                int(use_verbs), int(gt), *[x.data_ptr() for x in new], out.data_ptr(), gate.data_ptr(),
                _stream_ptr(self.device)))
        return (out, gate), new

    # ------------------------------------------------------------------ decode drivers
    def beam_search(self, beam_size, out_size, eos_idxs, use_verbs=False, gt=False,
                    trace_steps=False, forced=None):
        b, T, V = self.b, self.dims["seq_len"], self.dims["vocab_size"]
        dev = self.device
        words = torch.empty((b, out_size, T), device=dev, dtype=torch.long)
        gates = torch.empty((b, out_size, T), device=dev, dtype=torch.long)
        lpw = torch.empty((b, out_size, T), device=dev, dtype=torch.float32)
        lpg = torch.empty((b, out_size, T), device=dev, dtype=torch.float32)
        eos = (c_i64 * 2)(int(eos_idxs[0]), int(eos_idxs[1]))
        tr, tr_ref, extra = None, None, {}
        if trace_steps or forced is not None:
            tr = VsrTrace()
            if trace_steps:
                extra["step_out"] = torch.zeros((T, b * beam_size, V), device=dev)
                extra["step_gate"] = torch.zeros((T, b * beam_size, 2), device=dev)
                tr.step_out, tr.step_gate = extra["step_out"].data_ptr(), extra["step_gate"].data_ptr()
            if forced is not None:
                fb, fw, fg = [x.to(dev, torch.int32).contiguous() for x in forced]
                for x in (fb, fw, fg):
                    if tuple(x.shape) != (T, b, beam_size):
                        raise VsrError("forced selections must be (T, b, beam)")
                extra["_forced"] = (fb, fw, fg)
                tr.forced_beam, tr.forced_word, tr.forced_gate = fb.data_ptr(), fw.data_ptr(), fg.data_ptr()
            tr_ref = ctypes.byref(tr)
        with torch.cuda.device(dev):
            _lib.check(self.lib, self.lib.vsr_beam_search(
                self.handle, int(beam_size), int(out_size), eos, int(use_verbs), int(gt),
                words.data_ptr(), gates.data_ptr(), lpw.data_ptr(), lpg.data_ptr(), tr_ref,
                _stream_ptr(dev)))
        self._last = (T, b, beam_size)
        self._attn_shape = (b, out_size, T, self.R)
        return (words, gates), (lpw, lpg), extra

    def history(self):
        T, b, k = self._last
        dev = self.device
        parent, word, gate = [torch.empty((T, b, k), device=dev, dtype=torch.int32) for _ in range(3)]
        score = torch.empty((T, b, k), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            _lib.check(self.lib, self.lib.vsr_get_history(self.handle, parent.data_ptr(), word.data_ptr(),
                                                          gate.data_ptr(), score.data_ptr(), _stream_ptr(dev)))
        return parent, word, gate, score

    def forward_teacher(self, captions: torch.Tensor):
        _req_cuda(captions, "captions", torch.long)
        b, V = self.b, self.dims["vocab_size"]
        if captions.dim() != 2 or captions.size(0) != b:
            raise VsrError("captions must be (b, T)")
        T = captions.size(1)
        cap = captions.contiguous()
        out = torch.empty((b, T, V), device=self.device, dtype=torch.float32)
        gate = torch.empty((b, T, 2), device=self.device, dtype=torch.float32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_forward_teacher(self.handle, cap.data_ptr(), T, out.data_ptr(),
                                                              gate.data_ptr(), _stream_ptr(self.device)))
        self._attn_shape = (b, None, T, self.R)
        return out, gate

    def greedy(self):
        b, T = self.b, self.dims["seq_len"]
        words = torch.empty((b, T), device=self.device, dtype=torch.long)
        gates = torch.empty((b, T), device=self.device, dtype=torch.long)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_greedy(self.handle, words.data_ptr(), gates.data_ptr(),
                                                     _stream_ptr(self.device)))
        self._attn_shape = (b, None, T, self.R)
        return words, gates

    def sample(self, seed: int, n=1, temperature=1.0, top_k=0, top_p=1.0, use_verbs=False, gt=False):
        """Sampling decode (vsr_sample_ex): n independent draws per caption, the word head at `temperature`, truncated
        to the top_k most likely words (0 = off) and then to the smallest set of them holding top_p of their mass
        (1 = off); use_verbs / gt force verb slots as step_v does.  Returns (words, gates) int64 and (lp_words, lp_gates)
        fp32, shaped (b, T) when n == 1 and (b, n, T) otherwise; the log-probs are the model's own, untempered and
        untruncated.  Draw j of a caption is the same for every n > j.  The semantics are spelled out in
        include/vsrdec.h (vsr_sample_ex)."""
        check_sample_args(n, temperature, top_k, top_p, self.b)
        if use_verbs and (self._keep is None or self._keep[2] is None):
            raise VsrError("use_verbs needs a prologue with a verbs tensor")
        b, T = self.b, self.dims["seq_len"]
        shape = (b, T) if n == 1 else (b, int(n), T)
        words = torch.empty(shape, device=self.device, dtype=torch.long)
        gates = torch.empty(shape, device=self.device, dtype=torch.long)
        lpw = torch.empty(shape, device=self.device, dtype=torch.float32)
        lpg = torch.empty(shape, device=self.device, dtype=torch.float32)
        prm = VsrSampleParams(int(seed) & 0xFFFFFFFFFFFFFFFF, int(n), float(temperature), int(min(top_k, 2 ** 31 - 1)), float(top_p),
                              int(bool(use_verbs)), int(bool(gt)))
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_sample_ex(self.handle, ctypes.byref(prm), words.data_ptr(),
                                                        gates.data_ptr(), lpw.data_ptr(), lpg.data_ptr(),
                                                        _stream_ptr(self.device)))
        self._attn_shape = (b, None if n == 1 else int(n), T, self.R)
        return (words, gates), (lpw, lpg)

    # ------------------------------------------------------------------ attention capture
    def set_attention_capture(self, on: bool):
        """Record the per-step attention of the following decodes (vsr_set_attention_capture); off by default."""
        _lib.check(self.lib, self.lib.vsr_set_attention_capture(self.handle, int(bool(on))))

    def attention(self):
        """Attention of the last decode (vsr_get_attention): {"alpha": float32, "slot": int64}, shaped
        (b, out_size, T, R+1) / (b, out_size, T) after a beam search (following each returned beam's back-pointer
        path), (b, n, T, R+1) / (b, n, T) after sample(n > 1), (b, T, R+1) / (b, T) after the other drivers.  alpha[..., 0] is the sentinel, alpha[..., r+1] region r
        of the slot read at that step.  Raises VsrError when that decode ran without capture."""
        if self._attn_shape is None:
            raise VsrError("attention(): no decode has run on this engine")
        b, out_size, T, R = self._attn_shape
        lead = (b, T) if out_size is None else (b, out_size, T)
        alpha = torch.empty(lead + (R + 1,), device=self.device, dtype=torch.float32)
        slot = torch.empty(lead, device=self.device, dtype=torch.int32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib, self.lib.vsr_get_attention(self.handle, alpha.data_ptr(), slot.data_ptr(),
                                                            _stream_ptr(self.device)))
        return {"alpha": alpha, "slot": slot.long()}

    # ------------------------------------------------------------------ n-gram blocking
    def set_no_repeat_ngram(self, n: int):
        """Ban every word that would repeat an n-gram of the row's own words in the following beam-search, greedy and
        sampling decodes (vsr_set_no_repeat_ngram); 0 = off, the default.  n is an int in [0, seq_len]."""
        check_no_repeat_ngram(n, self.dims["seq_len"])
        _lib.check(self.lib, self.lib.vsr_set_no_repeat_ngram(self.handle, int(n)))
        self.no_repeat_ngram = int(n)

    # ------------------------------------------------------------------ diverse beam search
    def set_beam_diversity(self, groups: int, penalty: float):
        """Split the following beam searches into `groups` groups of beam_size / groups beams, each penalised by
        `penalty` per earlier group's pick of the same word at the step (vsr_set_beam_diversity); groups = 1 is off,
        the default.  The beam scores stay the model's."""
        check_beam_diversity(groups, penalty)
        _lib.check(self.lib, self.lib.vsr_set_beam_diversity(self.handle, int(groups), float(penalty)))
        self.beam_diversity = (int(groups), float(penalty))

    # ------------------------------------------------------------------ instrumentation
    def launch_count(self) -> int:
        return int(self.lib.vsr_launch_count(self.handle))

    def gemm_kind(self) -> str:
        return self.lib.vsr_gemm_kind(self.handle).decode()

    def set_profiling(self, on: bool):
        _lib.check(self.lib, self.lib.vsr_set_profiling(self.handle, int(on)))

    def step_times(self):
        """ms of every decoder step of the last profiled beam search (CUDA events between the steps)."""
        cap = 512
        ms = (c_f * cap)()
        with torch.cuda.device(self.device):
            n = self.lib.vsr_get_step_times(self.handle, ms, cap)
        if n < 0:
            _lib.check(self.lib, n)
        return [float(ms[i]) for i in range(n)]

    def phase_times(self):
        cap = 32
        names = (ctypes.c_char_p * cap)()
        ms = (c_f * cap)()
        cnt = (c_i32 * cap)()
        with torch.cuda.device(self.device):
            n = self.lib.vsr_get_phase_times(self.handle, names, ms, cnt, cap)
        if n < 0:
            _lib.check(self.lib, n)
        return [(names[i].decode(), float(ms[i]), int(cnt[i])) for i in range(n)]
