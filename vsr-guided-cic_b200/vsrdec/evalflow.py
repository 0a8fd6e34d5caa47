"""The inner loop of the eval (coco_scripts/eval_coco.py:117-249) as one pipelined object: for every batch of captions the
role-ordering pre-step (`vsrdec.preorder.RoleOrderer`), the permutation of the slot list, and the beam-search decode through the
index-form entry point — with the pre-step of batch i + 1 enqueued on a side stream while batch i decodes.

    flow = EvalFlow(model, RoleOrderer(re_sort_net, sinkhorn_net), eos_idxs=[eos, -1], beam_size=5, gt=True)
    for (words, gates), (lp_words, lp_gates) in flow.run(batches):      # device tensors, one tuple per batch, in order
        ...

A batch is a dict with the names of the eval loop: host arrays `control_verb (C, max_verb)`, `det_seqs_v`, `det_seqs_sr`
`(C, fixed_len, max_verb)`, `verb_list (C, fixed_len[, 1])`; CUDA tensors `detections (C, D, F)` (or one image's `(1, D, F)`
expanded over its captions), `slot_index (C, fixed_len, R) int32` (>= 0 detection row, -2 mean row, -1 padding: the index form of
`det_seqs_all`), `seqs_perm (C, fixed_len, 2352)` (the concatenated (vis, txt, pos) rows of eval_coco.py:146); optionally
`slot_valid (C, fixed_len)` (default: slots with at least one region index)."""
from typing import Iterable, Iterator

import torch

from .preorder import RoleOrderer, permute_slot_index


class EvalFlow:
    def __init__(self, model, orderer: RoleOrderer, eos_idxs, beam_size: int = 5, out_size: int = 1, gt: bool = True,
                 overlap: bool = True, no_repeat_ngram_size: int = 0, num_beam_groups: int = 1,
                 diversity_penalty: float = 0.0):
        """no_repeat_ngram_size: n-gram blocking of every decode (see CaptioningModel.beam_search; 0 = off).
        num_beam_groups, diversity_penalty: diverse beam search of every decode (see beam_search; 1 group = off)."""
        self.model, self.orderer = model, orderer
        self.no_repeat_ngram_size = no_repeat_ngram_size
        self.num_beam_groups, self.diversity_penalty = num_beam_groups, diversity_penalty
        self.eos_idxs, self.beam_size, self.out_size, self.gt = eos_idxs, beam_size, out_size, gt
        self.overlap = bool(overlap)
        self._side = None

    def _begin(self, b):
        sv = b.get("slot_valid")
        if sv is None:
            sv = (b["slot_index"] != -1).any(-1).cpu()
        return self.orderer.order_begin(b["control_verb"], b["det_seqs_v"], b["det_seqs_sr"], b["verb_list"], b["seqs_perm"], sv)

    def _decode(self, b, src, verbs):
        dev = b["slot_index"].device
        statics = (b["detections"], permute_slot_index(b["slot_index"], src), verbs.to(dev).double())
        return self.model.beam_search_v_indexed(statics, self.eos_idxs, self.beam_size, self.out_size, gt=self.gt,
                                                no_repeat_ngram_size=self.no_repeat_ngram_size,
                                                num_beam_groups=self.num_beam_groups,
                                                diversity_penalty=self.diversity_penalty)

    def run(self, batches: Iterable[dict]) -> Iterator:
        it = iter(batches)
        try:
            cur = next(it)
        except StopIteration:
            return
        if not self.overlap:
            while cur is not None:
                src, verbs = self.orderer.order_end(self._begin(cur))
                yield self._decode(cur, src, verbs)
                cur = next(it, None)
            return
        dev = cur["slot_index"].device
        if self._side is None or self._side.device != dev:
            self._side = torch.cuda.Stream(device=dev)
        main = torch.cuda.current_stream(dev)
        self._side.wait_stream(main)                          # the batch's tensors were produced on the caller's stream
        with torch.cuda.stream(self._side):
            state = self._begin(cur)
        while cur is not None:
            nxt = next(it, None)
            with torch.cuda.stream(self._side):
                src, verbs = self.orderer.order_end(state)    # host waits for this batch's pre-step only
                if nxt is not None:
                    self._side.wait_stream(main)
                    state = self._begin(nxt)                  # enqueued before the decode below: runs beside it
            yield self._decode(cur, src, verbs)
            cur = nxt
