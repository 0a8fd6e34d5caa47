"""Decode drivers of the captioning model, B200-native.

Same class surface as the reference's models/CaptioningModel.py:8-294 (`forward`, `test`,
`sample_rl`, `beam_search`, `beam_search_v`, `_select_beam[_i]`), but each driver hands the
WHOLE loop to libvsrdec (vsr_forward_teacher / vsr_greedy / vsr_sample / vsr_beam_search): the per-step
Python loop, the per-step statics gather, the full candidate sort and every host sync of the
reference are gone.  Sub-classes provide `_engine_for(statics, seqs, verbs)`.

Every driver takes `return_attention=False`.  When True the usual return value gets one more element, a dict with
`alpha` (float32, the token outputs' shape + R+1: column 0 = the adaptive sentinel's weight, column r+1 = region r of the
slot read at that step) and `slot` (int64, the token outputs' shape: that slot).  The weights are the ones that form the
attended feature (0 at padding regions), untouched by verb forcing and not masked after a caption's EOS.  For beam search
they follow each returned beam's back-pointer path, unlike the log-probs, which are in slot order as in the reference.

Every driver (`beam_search`, `beam_search_v`, `beam_search_v_indexed`, `forward`, `test`, `sample_rl`, `sample_v`, and `step` /
`step_v` of the sub-class) takes region features in float32, float16 or bfloat16, one dtype for the detections and the
slot tiles.  The kernels widen half-precision values to fp32 as they load them, so every output is bit-identical to that
of the same call on the features' float32 upcast; only the bytes read and copied halve.

Every driver that chooses words (`beam_search`, `beam_search_v`, `beam_search_v_indexed`, `test`, `sample_rl`, `sample_v`)
takes `no_repeat_ngram_size=0`.  With n >= 1 a word that would complete an n-gram the row (for beam search: the beam's
own word path) has already emitted is banned at that step: beam search keeps the exact top-k of the words that are not
banned, greedy takes the best of them, sampling drops banned words before temperature / top-k / top-p.  The returned
log-probs stay the model's own; verb-forced words are never blocked.  0 = off, bit-identical to a call without the
keyword.  The semantics and limits (n <= seq_len; vocab_size >= beam_size + seq_len - 1, or >= seq_len for greedy and
sampling) are spelled out in include/vsrdec.h, vsr_set_no_repeat_ngram.

The beam-search drivers (`beam_search`, `beam_search_v`, `beam_search_v_indexed`) take `num_beam_groups=1,
diversity_penalty=0.0`: diverse beam search (Vijayakumar et al., AAAI 2018).  With G = num_beam_groups > 1 the beam is
split into G groups of beam_size / G beams that choose in turn at every step; a group's candidate loses
diversity_penalty per pick of the same word by an earlier group at that step.  The penalty only steers the selection:
the beam scores and log-probs stay the model's, and the final ranking is over all beams (out_size = beam_size returns
every group's).  1 = off, bit-identical to a call without the keywords.  Semantics and limits (G in [1, 8] dividing
beam_size, a finite penalty >= 0): include/vsrdec.h, vsr_set_beam_diversity.
"""
import torch
from torch import nn


class CaptioningModel(nn.Module):
    def __init__(self, seq_len):
        self.seq_len = seq_len
        super().__init__()

    # ---- interface of the reference base class (CaptioningModel.py:13-20)
    def init_weights(self):
        raise NotImplementedError

    def init_state(self, b_s, device):
        raise NotImplementedError

    def step(self, t, state, prev_outputs, images, seqs, *args, mode='teacher_forcing'):
        raise NotImplementedError

    def _engine_for(self, statics, seqs=None):
        raise NotImplementedError

    def _check_ngram(self, no_repeat_ngram_size, beam_size=1):
        """VsrError unless the block size is valid for this model and a decode with beam_size rows per caption."""
        from vsrdec.engine import check_no_repeat_ngram
        check_no_repeat_ngram(no_repeat_ngram_size, self.seq_len, self.vocab_size, beam_size)

    @staticmethod
    def _check_diversity(num_beam_groups, diversity_penalty, beam_size):
        """VsrError unless the diverse beam search setting is valid for a beam search of beam_size."""
        from vsrdec.engine import check_beam_diversity
        check_beam_diversity(num_beam_groups, diversity_penalty, beam_size)

    @staticmethod
    def _run(eng, decode, return_attention, no_repeat_ngram_size=0, diversity=(1, 0.0)):
        """decode() alone, or with the engine's attention capture on around it: (result, attention dict or None).  The
        engine's n-gram blocking is no_repeat_ngram_size and its beam diversity (groups, penalty) is `diversity` for the
        duration of the call; both are restored afterwards."""
        prev, prev_div = eng.no_repeat_ngram, eng.beam_diversity
        if no_repeat_ngram_size != prev:
            eng.set_no_repeat_ngram(no_repeat_ngram_size)
        try:
            if tuple(diversity) != prev_div:
                eng.set_beam_diversity(*diversity)
            if not return_attention:
                return decode(), None
            eng.set_attention_capture(True)
            try:
                res = decode()
                att = eng.attention()
            finally:
                eng.set_attention_capture(False)
            return res, att
        finally:
            if eng.no_repeat_ngram != prev:
                eng.set_no_repeat_ngram(prev)
            if eng.beam_diversity != prev_div:
                eng.set_beam_diversity(*prev_div)

    # ---- drivers
    def forward(self, statics, seqs, *args, return_attention=False):
        """Teacher-forced unroll (reference CaptioningModel.py:22-36): returns
        (out (B,T,V), gate (B,T,2)) log-probabilities (+ attention (B,T,R+1), slot == t)."""
        eng = self._engine_for(statics, seqs)
        res, att = self._run(eng, lambda: eng.forward_teacher(seqs[0]), return_attention)
        return res if att is None else (*res, att)

    def test(self, statics, *args, return_attention=False, no_repeat_ngram_size=0):
        """Greedy decode (reference CaptioningModel.py:38-52): (words (b,T), gates (b,T)) (+ attention).  With
        no_repeat_ngram_size = n >= 1 each pick is the best word that does not repeat an n-gram of the caption."""
        self._check_ngram(no_repeat_ngram_size)
        eng = self._engine_for(statics)
        res, att = self._run(eng, eng.greedy, return_attention, no_repeat_ngram_size)
        return res if att is None else (*res, att)

    def sample_rl(self, statics, *args, seed=None, return_attention=False, n=1, temperature=1.0, top_k=0, top_p=1.0,
                  no_repeat_ngram_size=0):
        """Multinomial sampling with log-probs (reference CaptioningModel.py:54-76): at every step both heads are
        sampled from the step's distributions and fed back; returns ((words, gates), (lp_words, lp_gates)), each (b,T).
        The whole loop runs on the device (vsr_sample: Gumbel-max over the vocabulary row with a Philox stream).  The
        stream's seed is drawn from torch's CPU generator unless given, so torch.manual_seed() makes it reproducible
        (the draws differ from torch.distributions' — another generator — but follow the same distributions).
        Extensions (keywords only): n independent draws per caption, returned as (b, n, T) when n > 1 (draw j is the
        same for every n > j); the word head sampled at `temperature`, from its top_k most likely words (0 = off) and
        then from the smallest set of those that holds top_p of their mass (1 = off).  The log-probs stay the model's
        own (untempered, untruncated).  With no_repeat_ngram_size = m >= 1, words that would repeat an m-gram of the draw
        leave the row before temperature and truncation.  Semantics: include/vsrdec.h, vsr_sample_ex."""
        return self._sample(statics[:2], False, False, seed, return_attention, n, temperature, top_k, top_p,
                            no_repeat_ngram_size)

    def sample_v(self, statics, *, n=1, temperature=1.0, top_k=0, top_p=1.0, gt=False, seed=None, return_attention=False,
                 no_repeat_ngram_size=0):
        """sample_rl with verb forcing (step_v semantics, gt as in beam_search_v): statics = (detections, det_seqs,
        verbs).  A step whose slot holds a verb takes the forced word and gate 1, both with log-prob 0; the other steps
        are sampled as in sample_rl.  Same return structure as sample_rl."""
        if len(statics) < 3 or statics[2] is None:
            from vsrdec import VsrError
            raise VsrError("sample_v needs statics = (detections, det_seqs, verbs)")
        return self._sample(statics, True, gt, seed, return_attention, n, temperature, top_k, top_p, no_repeat_ngram_size)

    def _sample(self, statics, use_verbs, gt, seed, return_attention, n, temperature, top_k, top_p, no_repeat_ngram_size):
        from vsrdec.engine import check_sample_args
        check_sample_args(n, temperature, top_k, top_p, statics[0].size(0))   # before the prologue: nothing runs
        self._check_ngram(no_repeat_ngram_size)
        eng = self._engine_for(statics)
        if seed is None:
            seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        res, att = self._run(eng, lambda: eng.sample(seed, n=n, temperature=temperature, top_k=top_k, top_p=top_p,
                                                     use_verbs=use_verbs, gt=gt), return_attention, no_repeat_ngram_size)
        return res if att is None else (*res, att)

    def _select_beam(self, input, selected_beam, cur_beam_size, beam_size, b_s, reduced=True):
        """Beam-axis gather over (nested) tensors (reference CaptioningModel.py:78-94).  Kept for
        API compatibility; the device path never copies statics per beam."""
        if not isinstance(input, (list, tuple)):
            return self._select_beam_i(input, selected_beam, cur_beam_size, beam_size, b_s, reduced=reduced)
        picked = []
        for s in input:
            if isinstance(s, (list, tuple)):
                picked.append(tuple(self._select_beam_i(ss, selected_beam, cur_beam_size, beam_size, b_s,
                                                        reduced=reduced) for ss in s))
            else:
                picked.append(self._select_beam_i(s, selected_beam, cur_beam_size, beam_size, b_s,
                                                  reduced=reduced))
        return picked

    def _select_beam_i(self, input, selected_beam, cur_beam_size, beam_size, b_s, reduced=True):
        """(reference CaptioningModel.py:96-114)"""
        tail = tuple(input.shape[1:] if reduced else input.shape[2:])
        src = input.reshape((b_s, cur_beam_size) + tail)
        rows = torch.arange(b_s, device=input.device).unsqueeze(1)
        out = src[rows, selected_beam.long().reshape(b_s, beam_size)]
        return out.reshape((b_s * beam_size,) + tail) if reduced else out

    def _beam_run(self, eng, eos_idxs, beam_size, out_size, use_verbs, gt, return_attention, slot_index=None,
                  no_repeat_ngram_size=0, diversity=(1, 0.0)):
        def decode():
            return eng.beam_search(beam_size, out_size, eos_idxs, use_verbs=use_verbs, gt=gt)
        ((words, gates), (lpw, lpg), _), att = self._run(eng, decode, return_attention, no_repeat_ngram_size, diversity)
        outputs, log_probs = [words, gates], [lpw, lpg]
        if att is not None and slot_index is not None:      # detection row of every region of the slot read
            b, R = slot_index.size(0), slot_index.size(2)
            idx = att["slot"].reshape(b, -1, 1).expand(-1, -1, R)
            att["det_index"] = torch.gather(slot_index.long(), 1, idx).reshape(att["slot"].shape + (R,))
        if out_size == 1:
            outputs = [o.squeeze(1) for o in outputs]
            log_probs = [lp.squeeze(1) for lp in log_probs]
            if att is not None:
                att = {k: v.squeeze(1) for k, v in att.items()}
        return (outputs, log_probs) if att is None else (outputs, log_probs, att)

    def _beam(self, statics, eos_idxs, beam_size, out_size, use_verbs, gt, return_attention=False, no_repeat_ngram_size=0,
              num_beam_groups=1, diversity_penalty=0.0):
        self._check_ngram(no_repeat_ngram_size, beam_size)
        self._check_diversity(num_beam_groups, diversity_penalty, beam_size)
        eng = self._engine_for(statics)
        return self._beam_run(eng, eos_idxs, beam_size, out_size, use_verbs, gt, return_attention,
                              no_repeat_ngram_size=no_repeat_ngram_size, diversity=(num_beam_groups, diversity_penalty))

    def beam_search_v_indexed(self, statics, eos_idxs, beam_size, out_size=1, *args, gt=False, return_attention=False,
                              no_repeat_ngram_size=0, num_beam_groups=1, diversity_penalty=0.0):
        """Extension (SURVEY §8 f3): beam_search_v with the slots given as INDICES into the detections instead
        of materialised feature tiles: statics = (detections (b,D,F), slot_index (b,L,R) int, verbs (b,L) or None);
        slot_index >= 0 picks a detection row, -2 the mean of the image's valid detections, -1 is padding.
        Same return structure as beam_search_v; 10x fewer input bytes.  With return_attention the attention dict also
        holds det_index (..., R) int64 = slot_index[caption, slot, :]: the detection row each alpha[..., 1:] column
        weighs (-2 the image's mean row, -1 padding).  no_repeat_ngram_size, num_beam_groups and diversity_penalty as in
        beam_search."""
        self._check_ngram(no_repeat_ngram_size, beam_size)
        self._check_diversity(num_beam_groups, diversity_penalty, beam_size)
        eng = self._engine()
        verbs = statics[2] if len(statics) > 2 else None
        eng.prologue_indexed(statics[0], statics[1], verbs)
        self._prologue_key = None
        return self._beam_run(eng, eos_idxs, beam_size, out_size, verbs is not None, gt, return_attention,
                              slot_index=statics[1], no_repeat_ngram_size=no_repeat_ngram_size,
                              diversity=(num_beam_groups, diversity_penalty))

    def beam_search(self, statics, eos_idxs, beam_size, out_size=1, *args, return_attention=False, no_repeat_ngram_size=0,
                    num_beam_groups=1, diversity_penalty=0.0):
        """Joint (word, gate) beam search (reference CaptioningModel.py:116-195).  beam_size <= 8, out_size <= beam_size,
        <= 64 regions per slot (see the limits in models/controllable_captioning.py).  With no_repeat_ngram_size = n >= 1
        no beam picks a word that would repeat an n-gram of its own word path (the scores stay the model's).  With
        num_beam_groups = G > 1 the search is a diverse beam search of G groups, diversity_penalty per earlier group's
        pick of the same word (see the module docstring)."""
        return self._beam(statics[:2], eos_idxs, beam_size, out_size, False, False, return_attention, no_repeat_ngram_size,
                          num_beam_groups, diversity_penalty)

    def beam_search_v(self, statics, eos_idxs, beam_size, out_size=1, *args, gt=False, return_attention=False,
                      no_repeat_ngram_size=0, num_beam_groups=1, diversity_penalty=0.0):
        """Beam search with verb forcing (reference CaptioningModel.py:197-294).  beam_size <= 8, out_size <= beam_size,
        <= 64 regions per slot (see the limits in models/controllable_captioning.py).  no_repeat_ngram_size,
        num_beam_groups and diversity_penalty as in beam_search; a verb-forced word is never blocked or penalised."""
        return self._beam(statics, eos_idxs, beam_size, out_size, True, gt, return_attention, no_repeat_ngram_size,
                          num_beam_groups, diversity_penalty)
