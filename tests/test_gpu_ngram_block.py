"""No-repeat n-gram blocking in the beam-search, greedy and sampling decodes (vsr_set_no_repeat_ngram, the
`no_repeat_ngram_size` keyword of the drivers).

The reference for the ban is `banned` below, a plain restatement of the rule in include/vsrdec.h, applied along the
DEVICE's own trajectory: the oracle's `decoder_step` / `beam_search(forced=...)` recompute every step's log-probs on the
CPU, and each device choice must be a valid choice among the words that are not banned, up to the tie band of
tests/common.py: verify_device_beam.

GPU tests are marked one by one: the CPU-only cases at the end run without a device."""
import os
import subprocess
import sys

import pytest
import torch

from oracle import vsr_oracle as O
from common import load_golden, rel_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
REL, ABS = 1e-3, 1e-4
BAND_ABS, BAND_REL = 2e-3, 1e-4        # verify_device_beam's tie band


def _cuda(*ts):
    return tuple(t.to(DEV) if t is not None else None for t in ts)


def banned(y, n):
    """Words banned after the emitted words y (a list) with block size n: y[i + n - 1] for every start
    0 <= i <= len(y) - n whose n - 1 words equal the last n - 1 words of y."""
    t = len(y)
    if n <= 0:
        return set()
    return {y[i + n - 1] for i in range(t - n + 1) if y[i:i + n - 1] == y[t - n + 1:t]}


def repeated_ngrams(y, n):
    """Positions p >= n - 1 whose n-gram y[p-n+1 .. p] already ended at an earlier position."""
    seen, out = set(), []
    for p in range(n - 1, len(y)):
        g = tuple(y[p - n + 1:p + 1])
        if g in seen:
            out.append(p)
        seen.add(g)
    return out


def _forced_rows(out):
    """Rows of a step_v output that a verb forces: 0 at one word, -1e6 everywhere else."""
    return (out == 0).sum(1).eq(1) & (out == -1e6).sum(1).eq(out.size(1) - 1)


# ----------------------------------------------------------------------------- beam search against the oracle
def verify_blocked_beam(W, d, statics, eos, k, hist, n, use_verbs=False, gt=False, table=None):
    """Replay the device's beam trajectory through the oracle.  At every (step, caption), over the candidates whose word
    is not banned for its beam (verb-forced rows and beams frozen by the double-EOS path keep all of theirs):
      * every selected candidate is allowed and scores >= the k-th best allowed candidate - band;
      * every allowed candidate above the k-th best + band was selected;
      * the device's accumulated score is the oracle's at the selected candidate.
    Returns (decisions, number of steps at which some full beam had a banned word)."""
    parent, word, gate, score = [x.cpu().long() if x.dtype == torch.int32 else x.cpu() for x in hist]
    T, b, _ = parent.shape
    V = d.vocab_size
    forced = O.BeamTrace([parent[t] for t in range(T)], [word[t] for t in range(T)], [gate[t] for t in range(T)],
                         [], [], [], [])
    paths = [[[]] for _ in range(b)]                 # word path of every slot of the current step
    live = [torch.ones((b, 1)), torch.ones((b, 1))]  # sticky EOS masks of the current slots (t > 0)
    stats = {"decisions": 0, "bans": 0, "violations": []}

    def hook(t, out, gate_lp, flat):
        cur = flat.size(1) // (2 * V)
        full = (live[0] + live[1]).clamp(0, 1) != 0 if t > 0 else torch.ones((b, cur), dtype=torch.bool)
        frc = _forced_rows(out).view(b, cur) if use_verbs else torch.zeros((b, cur), dtype=torch.bool)
        allow = torch.ones((b, cur, V, 2), dtype=torch.bool)
        for c in range(b):
            for j in range(cur):
                ws = banned(paths[c][j], n)
                if ws and bool(full[c, j]) and not bool(frc[c, j]):
                    allow[c, j, list(ws), :] = False
                    stats["bans"] += 1
        allow = allow.view(b, -1)
        masked = torch.where(allow, flat, torch.full_like(flat, -float("inf")))
        sel = parent[t] * (2 * V) + word[t] * 2 + gate[t]
        sel_sc = flat.gather(1, sel)
        top = torch.topk(masked, k, dim=1).values
        kth = top[:, k - 1]
        band = BAND_ABS + BAND_REL * kth.abs()
        stats["decisions"] += b
        for c in range(b):
            if not bool(allow[c, sel[c]].all()):
                stats["violations"].append(f"t={t} caption={c}: a banned word was selected")
            if bool((sel_sc[c] < kth[c] - band[c]).any()):
                stats["violations"].append(f"t={t} caption={c}: selected {sel_sc[c].tolist()} below k-th {float(kth[c])}")
            must = (masked[c] > kth[c] + band[c]).nonzero().flatten().tolist()
            if not set(must) <= set(sel[c].tolist()):
                stats["violations"].append(f"t={t} caption={c}: a decisive allowed candidate was not selected")
            err = (score[t, c] - sel_sc[c]).abs()
            if bool((err > BAND_ABS + 2 * BAND_REL * sel_sc[c].abs()).any()):
                stats["violations"].append(f"t={t} caption={c}: score {score[t, c].tolist()} vs {sel_sc[c].tolist()}")
        # the next step's slots: parent's path + the picked word, sticky masks as CaptioningModel.py:143-144
        new_paths = [[paths[c][int(parent[t, c, j])] + [int(word[t, c, j])] for j in range(k)] for c in range(b)]
        paths[:] = new_paths
        pl = [x.gather(1, parent[t]) for x in live]
        live[0] = pl[0] * (word[t] != eos[0]).float()
        live[1] = pl[1] * (gate[t] != eos[1]).float()

    with torch.no_grad():
        O.beam_search(W, d, statics, eos, k, k, use_verbs=use_verbs, gt=gt, verb_table=table, forced=forced,
                      step_hook=hook)
    return stats


def _device_beam(m, statics, eos, k, n, use_verbs, gt, trace=False):
    eng = m._engine_for(_cuda(*statics))
    eng.set_no_repeat_ngram(n)
    try:
        (w, g), (lw, lg), extra = eng.beam_search(k, 1, eos, use_verbs=use_verbs, gt=gt, trace_steps=trace)
        hist = eng.history()
    finally:
        eng.set_no_repeat_ngram(0)
    torch.cuda.synchronize()
    return (w, g, lw, lg), hist, extra


GOLDEN_CASES = [("bs", False, False), ("bsv_gt", True, True), ("bsv_tab", True, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small_a.pt", "small_b.pt"])
@pytest.mark.parametrize("n", [1, 2, 3])
def test_beam_against_oracle_goldens(name, n):
    from gpu_common import make_model
    fx = load_golden(name)
    d, W = fx["dims_obj"], fx["weights"]
    m = make_model(d, W, fx["verb_table"])
    det, ds = fx["det"], fx["det_seqs"]
    for case, use_verbs, gt in GOLDEN_CASES:
        statics = (det, ds) if not use_verbs else (det, ds, fx["verbs_gt"] if gt else fx["verbs_tab"])
        for eos, k in (([3, -1], 3), ([3, 1], 5)):
            _, hist, _ = _device_beam(m, statics, eos, k, n, use_verbs, gt)
            st = verify_blocked_beam(W, d, statics, eos, k, hist, n, use_verbs, gt, fx["verb_table"])
            print(name, case, n, eos, k, st["decisions"], st["bans"])
            assert not st["violations"], st["violations"][:5]
            assert st["bans"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("n,sharpen", [(1, None), (2, 100.0), (3, None), (3, 100.0)])
def test_beam_against_oracle_config2(n, sharpen):
    """Config-2 size (b = 100, beam 5, V = 10000), raw and x100-sharpened out_fc, beam_search_v with gt verbs."""
    from gpu_common import make_model
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    if sharpen:
        W["out_fc.weight"] = W["out_fc.weight"] * sharpen
    m = make_model(d, W)
    statics = O.synth_inputs(100, 50, 10, 20, 2048, seed=1002, vocab_size=d.vocab_size, n_det_range=(10, 50),
                             verb_slots=(2,), verb_vocab_id=17)
    _, hist, _ = _device_beam(m, statics, [3, -1], 5, n, True, True)
    st = verify_blocked_beam(W, d, statics, [3, -1], 5, hist, n, True, True)
    print("config2", n, sharpen, st["decisions"], st["bans"])
    assert not st["violations"], st["violations"][:5]
    assert st["bans"] > 0


# ----------------------------------------------------------------------------- off is unchanged
def _small_a():
    from gpu_common import make_model
    fx = load_golden("small_a.pt")
    return fx, make_model(fx["dims_obj"], fx["weights"], fx["verb_table"])


def _flat(res):
    out = []
    for x in res:
        out.extend(_flat(x) if isinstance(x, (list, tuple)) else [x])
    return out


@pytest.mark.gpu
def test_off_is_unchanged():
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"], fx["verbs_gt"])
    eng = m._engine()
    calls = [
        lambda **kw: m.beam_search_v(dev, [3, -1], 3, 1, gt=True, **kw),
        lambda **kw: m.beam_search(dev[:2], [3, 1], 4, 2, **kw),
        lambda **kw: m.test(*dev[:2], **kw),
        lambda **kw: m.sample_rl(*dev[:2], seed=5, n=3, top_p=0.9, **kw),
    ]
    changed = []
    for call in calls:
        base = []
        for kw in (dict(), dict(no_repeat_ngram_size=0), dict(), dict(no_repeat_ngram_size=0)):   # 2nd / 3rd: graphs
            l0 = eng.launch_count()
            res = _flat(call(**kw))
            torch.cuda.synchronize()
            base.append((res, eng.launch_count() - l0))
        for res, launches in base[1:]:
            assert launches == base[0][1]
            assert all(torch.equal(x, y) for x, y in zip(res, base[0][0]))
        on = _flat(call(no_repeat_ngram_size=2))
        assert eng.no_repeat_ngram == 0
        changed.append(any(not torch.equal(x, y) for x, y in zip(on, base[0][0])))
        for _ in range(3):                                                       # off again: eager, capture, replay
            l0 = eng.launch_count()
            res = _flat(call())
            torch.cuda.synchronize()
            assert eng.launch_count() - l0 == base[0][1]
            assert all(torch.equal(x, y) for x, y in zip(res, base[0][0]))
    assert changed[2], changed          # greedy on small_a repeats itself, so blocking changes it (not vacuous)


# ----------------------------------------------------------------------------- blocking bites
def _assert_blocked(words, n):
    """No caption repeats an n-gram."""
    for c, y in enumerate(words.reshape(-1, words.shape[-1]).tolist()):
        assert not repeated_ngrams(y, n), (c, n, y)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3])
def test_blocking_bites_on_both_topk_paths(n):
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"])
    (w0, _), _ = m.beam_search(dev, [3, -1], 3, 3)
    assert any(repeated_ngrams(y, n) for y in w0.reshape(-1, w0.shape[-1]).tolist())    # not vacuous
    (w, g), (lw, lg) = m.beam_search(dev, [3, -1], 3, 3, no_repeat_ngram_size=n)
    _assert_blocked(w.cpu(), n)
    # the full-row kernel (k_softmax_topk, trace) selects exactly what the fused head (k_vocab_merge) selects
    (wf, gf, _, _), hf, _ = _device_beam(m, (fx["det"], fx["det_seqs"]), [3, -1], 3, n, False, False, trace=False)
    (wt, gt_, _, _), ht, extra = _device_beam(m, (fx["det"], fx["det_seqs"]), [3, -1], 3, n, False, False, trace=True)
    for x, y in zip(hf[:3], ht[:3]):                # parent, word, gate of every step
        assert torch.equal(x, y)
    assert torch.equal(wf, wt) and torch.equal(gf, gt_)
    # traced rows stay the model's full log-softmax (banned words included)
    assert bool(torch.isfinite(extra["step_out"]).all())


@pytest.mark.gpu
def test_blocking_with_verb_forcing():
    """Verb-forced words are never blocked; every other repeated n-gram is."""
    fx, m = _small_a()
    verbs = fx["verbs_gt"]
    dev = _cuda(fx["det"], fx["det_seqs"], verbs)
    for n in (1, 2):
        (w, g), _ = m.beam_search_v(dev, [3, -1], 3, 2, gt=True, no_repeat_ngram_size=n)
        (w1, g1), _ = m.sample_v(dev, n=4, gt=True, seed=3, no_repeat_ngram_size=n)
        for words, gates in ((w.cpu(), g.cpu()), (w1.cpu(), g1.cpu())):
            T = words.shape[-1]
            words, gates = words.reshape(-1, T), gates.reshape(-1, T)
            per = words.shape[0] // verbs.size(0)
            for r in range(words.shape[0]):
                # replay the slot pointer: slot_t = clamp(slot_{t-1} + gate_{t-1}); verb slots force their verb id
                slot, forced = 0, set()
                for t in range(T):
                    if t > 0:
                        slot = min(max(slot + int(gates[r, t - 1]), 0), verbs.size(1) - 1)
                    if int(verbs[r // per, slot]) != -1:
                        forced.add(t)
                y = words[r].tolist()
                bad = [p for p in repeated_ngrams(y, n) if p not in forced]
                assert not bad, (n, r, y, bad, forced)


@pytest.mark.gpu
def test_ffma_twin_subprocess():
    """VSRDEC_GEMM=simt (k_softmax_topk on every step): the blocked beam search passes the oracle check too."""
    code = ("import sys; sys.path[:0] = ['tests', '.', 'vsr-guided-cic_b200']\n"
            "import test_gpu_ngram_block as M\n"
            "from common import load_golden\n"
            "from gpu_common import make_model\n"
            "fx = load_golden('small_a.pt'); d, W = fx['dims_obj'], fx['weights']\n"
            "m = make_model(d, W, fx['verb_table'])\n"
            "assert m._engine().gemm_kind() == 'simt-fp32'\n"
            "st_all = []\n"
            "for n in (1, 2, 3):\n"
            "    st = (fx['det'], fx['det_seqs'], fx['verbs_tab'])\n"
            "    _, hist, _ = M._device_beam(m, st, [3, -1], 4, n, True, False)\n"
            "    s = M.verify_blocked_beam(W, d, st, [3, -1], 4, hist, n, True, False, fx['verb_table'])\n"
            "    assert not s['violations'] and s['bans'] > 0, s['violations'][:3]\n"
            "    w, _ = m.test(fx['det'].cuda(), fx['det_seqs'].cuda(), no_repeat_ngram_size=n)\n"
            "    M._assert_blocked(w.cpu(), n)\n"
            "print('simt ok')\n")
    env = dict(os.environ, VSRDEC_GEMM="simt")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "simt ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ----------------------------------------------------------------------------- greedy and sampling
def _replay(W, d, statics, words, gates, reps):
    """The oracle's per-step log-probs along the device's rows (caption-major, reps rows per caption)."""
    stat = tuple(s.repeat_interleave(reps, 0) for s in statics)
    N, T = words.shape
    state = O.init_state(d, N)
    prev, outs = None, []
    with torch.no_grad():
        for t in range(T):
            (out, _), state = O.decoder_step(W, d, t, state, prev, stat, None, "feedback")
            outs.append(out.double())
            prev = (words[:, t], gates[:, t])
    return torch.stack(outs)


def _allowed_mask(words, t, n, V):
    mask = torch.ones((words.shape[0], V), dtype=torch.bool)
    for r in range(words.shape[0]):
        ws = banned(words[r, :t].tolist(), n)
        if ws:
            mask[r, list(ws)] = False
    return mask


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 2, 3])
def test_greedy_picks_the_best_allowed_word(n):
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    statics = (fx["det"], fx["det_seqs"])
    w, g = m.test(*_cuda(*statics), no_repeat_ngram_size=n)
    w, g = w.cpu(), g.cpu()
    outs = _replay(W, d, statics, w, g, 1)
    n_top_banned = 0
    for t in range(d.seq_len):
        allow = _allowed_mask(w, t, n, d.vocab_size)
        lp = torch.where(allow, outs[t], torch.full_like(outs[t], -float("inf")))
        best = lp.max(1).values
        got = outs[t].gather(1, w[:, t:t + 1]).squeeze(1)
        assert bool(allow.gather(1, w[:, t:t + 1]).all()), t
        assert bool((got >= best - (BAND_ABS + BAND_REL * best.abs())).all()), t
        n_top_banned += int((~allow.gather(1, outs[t].argmax(1, keepdim=True))).sum())
    assert n_top_banned > 0
    _assert_blocked(w, n)


@pytest.mark.gpu
def test_sampling_exact_cases():
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    statics = (fx["det"], fx["det_seqs"])
    dev = _cuda(*statics)
    V, T = d.vocab_size, d.seq_len
    # top_k = 1: the best allowed word, also where the model's best word is banned
    for n in (1, 2, 3):
        (w, g), (lw, lg) = m.sample_rl(*dev, seed=4, n=3, top_k=1, no_repeat_ngram_size=n)
        w, g, lw = (x.cpu().reshape(-1, T) for x in (w, g, lw))
        outs = _replay(W, d, statics, w, g, 3)
        hits = 0
        for t in range(T):
            allow = _allowed_mask(w, t, n, V)
            lp = torch.where(allow, outs[t], torch.full_like(outs[t], -float("inf")))
            best = lp.max(1).values
            got = outs[t].gather(1, w[:, t:t + 1]).squeeze(1)
            assert bool(allow.gather(1, w[:, t:t + 1]).all())
            assert bool((got >= best - 1e-4 * best.abs() - 1e-5).all()), t
            assert rel_close(lw[:, t], got, REL, ABS)                   # the model's own log-prob
            hits += int((~allow.gather(1, outs[t].argmax(1, keepdim=True))).sum())
        assert hits > 0, n
        _assert_blocked(w, n)
    # plain and top-p draws: never banned, log-probs the model's, draw j the same for every number of draws
    for kw in (dict(), dict(top_p=0.9), dict(temperature=0.7, top_k=20)):
        for n in (1, 3, 5):
            full = m.sample_rl(*dev, seed=8, n=5, no_repeat_ngram_size=n, **kw)
            (w, g), (lw, lg) = full
            wc, gc, lwc = (x.cpu().reshape(-1, T) for x in (w, g, lw))
            _assert_blocked(wc, n)
            outs = _replay(W, d, statics, wc, gc, 5)
            for t in range(T):
                assert rel_close(lwc[:, t], outs[t].gather(1, wc[:, t:t + 1]).squeeze(1), REL, ABS)
            for j in (1, 3):
                part = m.sample_rl(*dev, seed=8, n=j, no_repeat_ngram_size=n, **kw)
                for x, y in zip(full[0] + full[1], part[0] + part[1]):
                    y = y.unsqueeze(1) if j == 1 else y
                    assert torch.equal(x[:, :j], y), (kw, n, j)


# ----------------------------------------------------------------------------- independence
@pytest.mark.gpu
def test_stacked_decode_equals_its_parts_and_pipeline():
    """1000 captions in one decode (CTA-pair GEMMs) equal ten 100-caption decodes bit for bit; DecodePipeline with the
    keyword equals direct calls."""
    from gpu_common import make_model
    from vsrdec import DecodePipeline
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    W["out_fc.weight"] = W["out_fc.weight"] * 100.0
    m = make_model(d, W)
    parts = [O.synth_inputs(100, 50, 10, 20, 2048, seed=1002 + i, vocab_size=d.vocab_size, n_det_range=(10, 50),
                            verb_slots=(2,), verb_vocab_id=17) for i in range(10)]
    big = tuple(torch.cat([p[i] for p in parts]) for i in range(3))
    ref = [m.beam_search_v(_cuda(*p), [3, -1], 5, 1, gt=True, no_repeat_ngram_size=3) for p in parts]
    (wb, gb), (lwb, lgb) = m.beam_search_v(_cuda(*big), [3, -1], 5, 1, gt=True, no_repeat_ngram_size=3)
    for i, ((w, g), (lw, lg)) in enumerate(ref):
        s = slice(100 * i, 100 * (i + 1))
        assert torch.equal(w, wb[s]) and torch.equal(g, gb[s]) and torch.equal(lw, lwb[s]) and torch.equal(lg, lgb[s]), i
    (w0, _), _ = m.beam_search_v(_cuda(*parts[0]), [3, -1], 5, 1, gt=True)
    assert not torch.equal(w0, ref[0][0][0])
    pipe = DecodePipeline([m], [3, -1], 5, 1, gt=True, stack=2, no_repeat_ngram_size=3)
    host = [tuple(t.pin_memory() for t in p) for p in parts[:4]]
    for i, (w, g, lw, lg) in enumerate(pipe.run(host)):
        assert torch.equal(w, ref[i][0][0].cpu()) and torch.equal(lw, ref[i][1][0].cpu()), i


# ----------------------------------------------------------------------------- errors
@pytest.mark.gpu
def test_invalid_arguments_raise_before_anything_runs():
    from vsrdec import VsrError
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"], fx["verbs_gt"])
    m.test(*dev[:2])
    eng = m._engine()
    torch.cuda.synchronize()
    l0 = eng.launch_count()
    T = fx["dims_obj"].seq_len
    for bad in (-1, T + 1, True, 1.0, "2", None):
        for call in (lambda: m.beam_search(dev[:2], [3, -1], 3, no_repeat_ngram_size=bad),
                     lambda: m.beam_search_v(dev, [3, -1], 3, gt=True, no_repeat_ngram_size=bad),
                     lambda: m.test(*dev[:2], no_repeat_ngram_size=bad),
                     lambda: m.sample_rl(*dev[:2], seed=1, no_repeat_ngram_size=bad),
                     lambda: m.sample_v(dev, seed=1, no_repeat_ngram_size=bad),
                     lambda: eng.set_no_repeat_ngram(bad)):
            with pytest.raises(VsrError):
                call()
    assert eng.launch_count() == l0 and eng.no_repeat_ngram == 0
    assert eng.lib.vsr_set_no_repeat_ngram(eng.handle, -1) == -1
    assert eng.lib.vsr_set_no_repeat_ngram(eng.handle, T + 1) == -1
    # a vocabulary too small for the beam: the library refuses too
    from gpu_common import make_model
    d = O.Dims(seq_len=8, vocab_size=10, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    ms = make_model(d, O.init_weights(d, seed=5))
    det, ds, _ = O.synth_inputs(3, 9, 5, 6, 64, seed=41, vocab_size=10, n_det_range=(3, 9), real_slots=(2, 5))
    with pytest.raises(VsrError):
        ms.beam_search(_cuda(det, ds), [3, -1], 4, no_repeat_ngram_size=2)          # 10 < 4 + 8 - 1
    e2 = ms._engine()
    e2.prologue(*_cuda(det, ds))
    e2.set_no_repeat_ngram(2)
    from vsrdec._lib import c_i64
    out = [torch.empty((3, 1, 8), device=DEV, dtype=dt) for dt in (torch.long, torch.long, torch.float32, torch.float32)]
    eos = (c_i64 * 2)(3, -1)
    assert e2.lib.vsr_beam_search(e2.handle, 4, 1, eos, 0, 0, *[x.data_ptr() for x in out], None, None) == -1
    assert e2.lib.vsr_beam_search(e2.handle, 3, 1, eos, 0, 0, *[x.data_ptr() for x in out], None, None) == 0
    e2.set_no_repeat_ngram(0)
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- CPU-only
def test_banned_restatement():
    assert banned([5, 6, 5], 2) == {6}
    assert banned([5, 6, 5, 6], 3) == {5}
    assert banned([1, 2, 3], 1) == {1, 2, 3}
    assert banned([1, 2], 3) == set()
    assert banned([4, 4], 2) == {4}
    assert repeated_ngrams([1, 2, 1, 2], 2) == [3]


def test_argument_check_without_a_device():
    from vsrdec import VsrError
    from vsrdec.engine import check_no_repeat_ngram
    check_no_repeat_ngram(0, 20, 5, 8)                 # off: no vocabulary condition
    check_no_repeat_ngram(3, 20, 24, 5)
    check_no_repeat_ngram(20, 20, 20, 1)
    check_no_repeat_ngram(2, 20)
    for args in ((-1, 20, 10000, 5), (21, 20, 10000, 5), (True, 20, 10000, 5), (2.0, 20, 10000, 5), ("3", 20, 10000, 5),
                 (None, 20, 10000, 5), (3, 20, 23, 5), (1, 20, 19, 1)):
        with pytest.raises(VsrError):
            check_no_repeat_ngram(*args)


def test_signatures_and_binding():
    import inspect
    import re
    from models import ControllableCaptioningModel
    from models.CaptioningModel import CaptioningModel
    from vsrdec import DecodePipeline, EvalFlow, EXPORTED_SYMBOLS
    for fn in (CaptioningModel.beam_search, CaptioningModel.beam_search_v, CaptioningModel.beam_search_v_indexed,
               CaptioningModel.test, CaptioningModel.sample_rl, CaptioningModel.sample_v,
               ControllableCaptioningModel.test, ControllableCaptioningModel.sample_rl, DecodePipeline.__init__,
               EvalFlow.__init__):
        assert inspect.signature(fn).parameters["no_repeat_ngram_size"].default == 0, fn
    assert "vsr_set_no_repeat_ngram" in EXPORTED_SYMBOLS
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vsrdec.h")).read(), flags=re.S)
    assert re.search(r"int vsr_set_no_repeat_ngram\(vsr_handle h, int32_t n\);", src)


def test_model_rejects_bad_sizes_before_the_engine():
    """The drivers validate the keyword before they touch the engine (here: a CPU model, whose engine would raise a
    different error)."""
    from vsrdec import VsrError
    from models import ControllableCaptioningModel
    m = ControllableCaptioningModel(8, 10, 2, det_feat_size=8, input_encoding_size=4, rnn_size=4, att_size=4,
                                    verb_tables=({}, {}))
    det, ds = torch.zeros(2, 3, 8), torch.zeros(2, 4, 2, 8)
    for call in (lambda: m.beam_search((det, ds), [3, -1], 4, no_repeat_ngram_size=2),     # 10 < 4 + 8 - 1
                 lambda: m.test(det, ds, no_repeat_ngram_size=9),
                 lambda: m.sample_rl(det, ds, no_repeat_ngram_size=True)):
        with pytest.raises(VsrError, match="no_repeat_ngram_size"):
            call()
