"""Throughput-oriented host loop around the drop-in model's beam search (what `bench.py`'s end-to-end figure runs).

The reference decodes one batch at a time on the default stream and `.cpu()`s the result (eval_coco.py:245-249).
Consecutive batches are independent, and so are the captions inside a batch (every op of the decoder is row-wise and
the top-k is per caption), so this helper

* STACKS `stack` consecutive host batches along the caption axis into one device decode: the step GEMMs then run
  several waves of tiles per launch (epilogues overlap the next tile's main loop, the weights are streamed once per
  group instead of once per batch) and the latency-bound small kernels are paid once per group.  A stacked decode is
  bit-identical to separate decodes (tests/test_gpu_parity.py: test_properties_at_full_size, test_decode_pipeline_*);
* keeps `lanes` such decodes in flight, each on its own engine (a model replica with the same weights) and CUDA stream;
* fills `buffers` device input buffers from pinned host memory on a copy stream that runs ahead of the lanes;
* copies results to pinned host memory asynchronously and hands them out one decode later, per batch, in order.

Nothing here changes what a decode computes: every group goes through `beam_search_v` (or `beam_search_v_indexed`)
exactly as a direct call on the concatenated batch would."""
from typing import Callable, Iterable, Iterator, List, Optional, Sequence, Tuple

import torch


class DecodePipeline:
    def __init__(self, models: Sequence, eos_idxs, beam_size: int, out_size: int = 1, gt: bool = False,
                 indexed: bool = False, buffers: Optional[int] = None, stack: int = 1, ramp: bool = True,
                 post: Optional[Callable[[torch.Tensor], torch.Tensor]] = None, no_repeat_ngram_size: int = 0,
                 num_beam_groups: int = 1, diversity_penalty: float = 0.0):
        """models: one drop-in model per lane (same weights, same device).  `stack` host batches (of equal shapes) are
        decoded per call; with `ramp` the first group of a run holds a single batch, so that the first decode starts after
        one batch's host->device copy instead of `stack` of them (the un-overlapped pipeline fill of a short run).  `post` is
        applied to each batch's words tensor on the lane's stream (e.g. the all-gather of a caption-sharded job).
        `no_repeat_ngram_size` is passed to every decode (n-gram blocking, see beam_search; 0 = off), and so are
        `num_beam_groups` and `diversity_penalty` (diverse beam search, see beam_search; 1 group = off)."""
        if not models:
            raise ValueError("DecodePipeline needs at least one model")
        self.models = list(models)
        self.device = next(self.models[0].parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("DecodePipeline: the models must live on a CUDA device (no CPU fallback)")
        self.eos_idxs, self.beam_size, self.out_size, self.gt, self.indexed = eos_idxs, beam_size, out_size, gt, indexed
        self.post = post
        self.no_repeat_ngram_size = no_repeat_ngram_size
        self.num_beam_groups, self.diversity_penalty = num_beam_groups, diversity_penalty
        self.stack = max(1, int(stack))
        self.ramp = bool(ramp)
        self.n_lanes = len(self.models)
        self.n_buf = buffers if buffers is not None else 2 * self.n_lanes
        # results are staged per input slot and collected one decode late: with a single slot decode s+1 would overwrite
        # (and re-record the event of) decode s before it has been handed out
        if self.n_buf < max(2, self.n_lanes):
            raise ValueError("DecodePipeline needs at least two input buffers and at least one per lane")
        self.lanes = [torch.cuda.Stream(self.device) for _ in range(self.n_lanes)]
        self.copy_stream = torch.cuda.Stream(self.device)
        self._bufs: List[Optional[Tuple[torch.Tensor, ...]]] = [None] * self.n_buf
        self._pinned: List[Optional[Tuple[torch.Tensor, ...]]] = [None] * self.n_buf
        self._count = [0] * self.n_buf          # batches staged in the slot
        self._rows = [0] * self.n_buf           # captions per batch of the slot's group
        self._ready = [torch.cuda.Event() for _ in range(self.n_buf)]
        self._freed = [torch.cuda.Event() for _ in range(self.n_buf)]
        self._done = [torch.cuda.Event() for _ in range(self.n_buf)]

    # ------------------------------------------------------------------ pieces
    def _stage(self, slot: int, group: Sequence[Sequence[torch.Tensor]]):
        """H2D copies of a group of host batches into input buffer `slot` (stacked along dim 0) on the copy stream."""
        first = group[0]
        b = first[0].shape[0]
        for hb in group[1:]:
            if any(h.shape != f.shape or h.dtype != f.dtype for h, f in zip(hb, first)):
                raise ValueError("DecodePipeline: the batches of one stacked group must have equal shapes")
        want = [((self.stack * b,) + tuple(h.shape[1:]), h.dtype) for h in first]
        bufs = self._bufs[slot]
        if bufs is None or any(tuple(t.shape) != s or t.dtype != dt for t, (s, dt) in zip(bufs, want)):
            bufs = tuple(torch.empty(s, dtype=dt, device=self.device) for s, dt in want)
            for t in bufs:                                      # written on the copy stream, read on the lanes: a buffer
                t.record_stream(self.copy_stream)               # dropped later (shape change) must not be recycled early
                for ln in self.lanes:
                    t.record_stream(ln)
            self._bufs[slot] = bufs
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self._freed[slot])      # the decode that last read this buffer has finished
            for i, hb in enumerate(group):
                for d_t, h_t in zip(bufs, hb):
                    d_t[i * b:(i + 1) * b].copy_(h_t, non_blocking=True)
            self._ready[slot].record(self.copy_stream)
        self._count[slot], self._rows[slot] = len(group), b

    def _decode(self, step: int, slot: int):
        lane_id = step % self.n_lanes
        lane, model = self.lanes[lane_id], self.models[lane_id]
        n, b = self._count[slot], self._rows[slot]
        lane.wait_event(self._ready[slot])
        with torch.cuda.stream(lane):
            fn = model.beam_search_v_indexed if self.indexed else model.beam_search_v
            statics = tuple(t[:n * b] for t in self._bufs[slot])
            (words, gates), (lpw, lpg) = fn(statics, self.eos_idxs, self.beam_size, self.out_size, gt=self.gt,
                                            no_repeat_ngram_size=self.no_repeat_ngram_size,
                                            num_beam_groups=self.num_beam_groups, diversity_penalty=self.diversity_penalty)
            self._freed[slot].record(lane)
            if self.post is not None:
                words = torch.cat([self.post(words[i * b:(i + 1) * b]) for i in range(n)], 0)
            outs = (words, gates, lpw, lpg)
            pin = self._pinned[slot]
            if pin is None or any(p.shape != o.shape for p, o in zip(pin, outs)):
                pin = tuple(torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs)
                self._pinned[slot] = pin
            for p, o in zip(pin, outs):
                p.copy_(o, non_blocking=True)                   # device -> host read of the group's result
            self._done[slot].record(lane)

    def _collect(self, slot: int, n: int):
        self._done[slot].synchronize()
        outs = tuple(p.clone() for p in self._pinned[slot])
        return [tuple(o[i * (o.shape[0] // n):(i + 1) * (o.shape[0] // n)] for o in outs) for i in range(n)]

    # ------------------------------------------------------------------ the loop
    def run(self, host_batches: Iterable[Sequence[torch.Tensor]]) -> Iterator[Tuple[torch.Tensor, ...]]:
        """host_batches yields tuples of pinned host tensors: (detections, det_seqs, verbs) or, with indexed=True,
        (detections, slot_index, verbs).  Yields (words, gates, lp_words, lp_gates) host tensors per batch, in order."""
        cur = torch.cuda.current_stream(self.device)
        for ev in self._freed:
            ev.record(cur)
        it = iter(host_batches)
        ahead = self.n_buf - self.n_lanes + 1       # groups staged before the decode that needs them is enqueued
        staged = 0
        pending: List[Tuple[int, int]] = []         # (slot, batches) of decodes enqueued but not yet handed out
        exhausted = False

        def stage_next():
            nonlocal staged, exhausted
            if exhausted:
                return False
            group = []
            want = 1 if (self.ramp and staged == 0) else self.stack
            while len(group) < want:
                try:
                    group.append(next(it))
                except StopIteration:
                    exhausted = True
                    break
            if not group:
                return False
            self._stage(staged % self.n_buf, group)
            staged += 1
            return True

        for _ in range(ahead):
            stage_next()
        step = 0
        while step < staged:
            slot = step % self.n_buf
            self._decode(step, slot)
            pending.append((slot, self._count[slot]))   # (re-staging the slot later changes _count, not this entry)
            step += 1
            stage_next()
            if len(pending) > 1:                    # hand out the previous decode's results while this one runs
                yield from self._collect(*pending.pop(0))
        while pending:
            yield from self._collect(*pending.pop(0))
