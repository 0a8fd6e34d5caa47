"""Diverse beam search (vsr_set_beam_diversity, the `num_beam_groups` / `diversity_penalty` keywords of the beam-search
drivers).

The reference for the grouped selection is `group_keys` / `select_groups` below, a plain restatement of the rule in
include/vsrdec.h.  It is applied along the DEVICE's own trajectory: the oracle's `beam_search(forced=...)` recomputes
every step's candidate scores on the CPU, the counts of each group come from the device's picks of the earlier groups,
and every device pick must be a valid choice of its group up to the tie band of tests/common.py: verify_device_beam.

GPU tests are marked one by one: the CPU-only cases at the end run without a device."""
import os
import subprocess
import sys
from collections import Counter

import pytest
import torch

from oracle import vsr_oracle as O
from common import load_golden, check_returned_beams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
BAND_ABS, BAND_REL = 2e-3, 1e-4        # verify_device_beam's tie band


def _cuda(*ts):
    return tuple(t.to(DEV) if t is not None else None for t in ts)


def _forced_rows(out):
    """Rows of a step_v output that a verb forces: 0 at one word, -1e6 everywhere else."""
    return (out == 0).sum(1).eq(1) & (out == -1e6).sum(1).eq(out.size(1) - 1)


def banned(y, n):
    """Words that n-gram blocking bans after the emitted words y (include/vsrdec.h, vsr_set_no_repeat_ngram)."""
    t = len(y)
    if n <= 0:
        return set()
    return {y[i + n - 1] for i in range(t - n + 1) if y[i:i + n - 1] == y[t - n + 1:t]}


# ----------------------------------------------------------------------------- the rule, restated
def group_keys(flat, cur, V, g, B, lam, live, forced_rows, prev_picks):
    """Keys of group g's candidates for one caption: (rows, keys (len(rows), V, 2)).  flat = the caption's candidate
    scores sc (cur * V * 2, flat index j * 2V + w * 2 + gate); rows = the group's parents (every row at t = 0, when
    cur = 1); prev_picks = flat indices of the earlier groups' picks at this step.  key = fl(sc - fl(lam * cnt(w))) on
    the rows that are live and not verb-forced, sc elsewhere."""
    rows = list(range(cur)) if cur == 1 else list(range(g * B, (g + 1) * B))
    key = flat.view(cur, V, 2)[rows].clone()
    cnt = Counter(int(p) % (2 * V) // 2 for p in prev_picks if live[int(p) // (2 * V)])
    pen = [i for i, j in enumerate(rows) if live[j] and not forced_rows[j]]
    lam32 = torch.tensor(lam, dtype=torch.float32)
    for w, n in cnt.items():
        key[pen, w, :] = key[pen, w, :] - lam32 * n
    return rows, key


def select_groups(flat, cur, k, G, lam, live, forced_rows):
    """The k picks (flat indices, slot order) of a G-group diverse selection of one caption: groups in order, each takes
    the B = k / G candidates of its own rows with the largest key, ties by flat index ascending."""
    V = flat.numel() // (2 * cur)
    B = k // G
    picks = []
    for g in range(G):
        rows, key = group_keys(flat, cur, V, g, B, lam, live, forced_rows, picks)
        order = torch.sort(key.flatten(), descending=True, stable=True).indices[:B]
        picks += [rows[0] * 2 * V + int(i) for i in order]
    return picks


# ----------------------------------------------------------------------------- against the oracle
def verify_diverse_beam(W, d, statics, eos, k, G, lam, hist, use_verbs=False, gt=False, table=None, ngram=0):
    """Replay the device's trajectory through the oracle.  At every (step, caption, group g), with the counts taken
    from the device's picks of groups 0 .. g-1:
      * each pick of g comes from g's own parents and its key is >= g's B-th best key - band;
      * every candidate of g whose key is above the B-th best + band was picked;
      * the device's stored score is the oracle's sc at the pick (the model's score, not the key).
    With ngram > 0 the words n-gram blocking bans for a live, unforced beam leave its candidates first.
    Returns (stats, oracle outputs, oracle log-probs); stats["changed"] counts the (step, caption, group) decisions
    with a pick that the group's plain top-B (by sc) would not have taken, outside the band."""
    parent, word, gate, score = [x.cpu().long() if x.dtype == torch.int32 else x.cpu() for x in hist]
    T, b, _ = parent.shape
    V, B = d.vocab_size, k // G
    forced = O.BeamTrace([parent[t] for t in range(T)], [word[t] for t in range(T)], [gate[t] for t in range(T)],
                         [], [], [], [])
    live_m = [torch.ones((b, 1)), torch.ones((b, 1))]
    paths = [[[]] for _ in range(b)]
    stats = {"decisions": 0, "changed": 0, "violations": []}

    def hook(t, out, gate_lp, flat):
        cur = flat.size(1) // (2 * V)
        full = (live_m[0] + live_m[1]).clamp(0, 1) != 0 if t > 0 else torch.ones((b, cur), dtype=torch.bool)
        frc = _forced_rows(out).view(b, cur) if use_verbs else torch.zeros((b, cur), dtype=torch.bool)
        sel = parent[t] * (2 * V) + word[t] * 2 + gate[t]
        for c in range(b):
            fc = flat[c]
            if ngram > 0:
                fc = fc.clone().view(cur, V, 2)
                for j in range(cur):
                    ws = banned(paths[c][j], ngram)
                    if ws and bool(full[c, j]) and not bool(frc[c, j]):
                        fc[j, list(ws), :] = -float("inf")
                fc = fc.view(-1)
            live, frow = full[c].tolist(), frc[c].tolist()
            for g in range(G):
                stats["decisions"] += 1
                rows, key = group_keys(fc, cur, V, g, B, lam, live, frow, sel[c, :g * B].tolist())
                key = key.flatten()
                base = rows[0] * 2 * V
                mine = [int(s) - base for s in sel[c, g * B:(g + 1) * B]]
                if any(not 0 <= m < key.numel() for m in mine):
                    stats["violations"].append(f"t={t} c={c} g={g}: a pick outside the group's parents")
                    continue
                top = torch.topk(key, B)
                bth = float(top.values[B - 1])
                band = BAND_ABS + BAND_REL * abs(bth)
                got = key[mine]
                if bool((got < bth - band).any()):
                    stats["violations"].append(f"t={t} c={c} g={g}: picks {got.tolist()} below the B-th key {bth}")
                must = (key > bth + band).nonzero().flatten().tolist()
                if not set(must) <= set(mine):
                    stats["violations"].append(f"t={t} c={c} g={g}: a decisive candidate was not picked")
                raw = fc.view(cur, V, 2)[rows].flatten()
                sc = raw[mine]
                err = (score[t, c, g * B:(g + 1) * B] - sc).abs()
                if bool((err > BAND_ABS + 2 * BAND_REL * sc.abs()).any()):
                    stats["violations"].append(f"t={t} c={c} g={g}: score {score[t, c, g * B:(g + 1) * B].tolist()} "
                                               f"vs sc {sc.tolist()}")
                raw_bth = float(torch.topk(raw, B).values[B - 1])
                stats["changed"] += int(bool((sc < raw_bth - (BAND_ABS + BAND_REL * abs(raw_bth))).any()))
        paths[:] = [[paths[c][int(parent[t, c, j])] + [int(word[t, c, j])] for j in range(k)] for c in range(b)]
        pl = [x.gather(1, parent[t]) for x in live_m]
        live_m[0] = pl[0] * (word[t] != eos[0]).float()
        live_m[1] = pl[1] * (gate[t] != eos[1]).float()

    with torch.no_grad():
        outs, lps = O.beam_search(W, d, statics, eos, k, k, use_verbs=use_verbs, gt=gt, verb_table=table, forced=forced,
                                  step_hook=hook)
    return stats, outs, lps


def _device_beam(m, statics, eos, k, G, lam, use_verbs, gt, out_size=None, trace=False, ngram=0):
    """A beam search through the engine with the diversity setting on: (w, g, lw, lg), history, extra."""
    eng = m._engine_for(_cuda(*statics))
    eng.set_beam_diversity(G, lam)
    eng.set_no_repeat_ngram(ngram)
    try:
        (w, g), (lw, lg), extra = eng.beam_search(k, out_size or k, eos, use_verbs=use_verbs, gt=gt, trace_steps=trace)
        hist = eng.history()
    finally:
        eng.set_beam_diversity(1, 0.0)
        eng.set_no_repeat_ngram(0)
    torch.cuda.synchronize()
    return (w, g, lw, lg), hist, extra


def _check(tag, W, d, statics, eos, k, G, lam, m, use_verbs, gt, table=None, ngram=0):
    dev, hist, _ = _device_beam(m, statics, eos, k, G, lam, use_verbs, gt, ngram=ngram)
    st, o_outs, o_lps = verify_diverse_beam(W, d, statics, eos, k, G, lam, hist, use_verbs, gt, table, ngram)
    print(tag, k, G, lam, st["decisions"], st["changed"])
    assert not st["violations"], (tag, st["violations"][:5])
    check_returned_beams(tag, d, hist, k, dev, o_outs, o_lps)
    return st


GOLDEN_CASES = [("bs", False, False), ("bsv_gt", True, True), ("bsv_tab", True, False)]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["small_a.pt", "small_b.pt"])
@pytest.mark.parametrize("lam", [0.5, 2.0])
def test_against_oracle_goldens(name, lam):
    from gpu_common import make_model
    fx = load_golden(name)
    d, W = fx["dims_obj"], fx["weights"]
    m = make_model(d, W, fx["verb_table"])
    det, ds = fx["det"], fx["det_seqs"]
    changed = 0
    for case, use_verbs, gt in GOLDEN_CASES:
        statics = (det, ds) if not use_verbs else (det, ds, fx["verbs_gt"] if gt else fx["verbs_tab"])
        for (k, G), eos in (((4, 2), [3, -1]), ((6, 3), [3, 1]), ((5, 5), [3, -1])):
            changed += _check(f"{name}/{case}", W, d, statics, eos, k, G, lam, m, use_verbs, gt,
                              fx["verb_table"])["changed"]
    assert changed > 0                      # the penalty changed some group's picks: the check is not vacuous


@pytest.mark.gpu
@pytest.mark.parametrize("sharpen", [None, 100.0])
def test_against_oracle_config2(sharpen):
    """Config-2 size (b = 100, V = 10000), beam 6 in 3 groups, raw and x100-sharpened out_fc, beam_search_v with gt
    verbs."""
    from gpu_common import make_model
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    if sharpen:
        W["out_fc.weight"] = W["out_fc.weight"] * sharpen
    m = make_model(d, W)
    statics = O.synth_inputs(100, 50, 10, 20, 2048, seed=1002, vocab_size=d.vocab_size, n_det_range=(10, 50),
                             verb_slots=(2,), verb_vocab_id=17)
    st = _check(f"config2 x{sharpen}", W, d, statics, [3, -1], 6, 3, 2.0 if sharpen else 0.5, m, True, True)
    assert st["changed"] > 0


@pytest.mark.gpu
def test_against_oracle_with_ngram_blocking():
    from gpu_common import make_model
    fx = load_golden("small_a.pt")
    d, W = fx["dims_obj"], fx["weights"]
    m = make_model(d, W, fx["verb_table"])
    st = _check("small_a/ngram3", W, d, (fx["det"], fx["det_seqs"]), [3, -1], 6, 3, 1.0, m, False, False, ngram=3)
    assert st["changed"] > 0
    # the keywords compose on the drivers too: no returned caption repeats a trigram
    (w, _), _ = m.beam_search(_cuda(fx["det"], fx["det_seqs"]), [3, -1], 6, 6, no_repeat_ngram_size=3,
                              num_beam_groups=3, diversity_penalty=1.0)
    for y in w.cpu().reshape(-1, d.seq_len).tolist():
        grams = [tuple(y[p - 2:p + 1]) for p in range(2, len(y))]
        assert len(grams) == len(set(grams)), y


# ----------------------------------------------------------------------------- lambda = 0 reduces exactly
def _config2_parts(n):
    return [O.synth_inputs(100, 50, 10, 20, 2048, seed=1002 + i, vocab_size=10000, n_det_range=(10, 50),
                           verb_slots=(2,), verb_vocab_id=17) for i in range(n)]


@pytest.mark.gpu
@pytest.mark.parametrize("captions", [100, 1000])
def test_zero_penalty_is_independent_searches(captions):
    """With lambda = 0 every group is a plain beam search of beam B = k / G, bit for bit (rows are bit-independent,
    DESIGN.md §2), with one exactly characterised exception.  fl(seq + fl(word + gate)) can round two words of one row
    to the SAME score.  The flat-index rule then prefers the lower word index; a group sees its rows' top-k words and
    applies it, while the plain search of beam B only holds its rows' top-B words and can miss the lower-index one
    (DESIGN.md §2).  At the first step where a caption's group and its plain search part, both picks must have that
    bit-identical score, the same parent and gate, and the group's word must be the lower index; every other caption
    must match bit for bit at every step."""
    from gpu_common import make_model
    d = O.Dims()
    m = make_model(d, O.init_weights(d, seed=1234))
    parts = _config2_parts(captions // 100)
    statics = tuple(torch.cat([p[i] for p in parts]) for i in range(3))
    for k, G in ((6, 3), (6, 2), (4, 4)):
        B = k // G
        tied = set()
        _, hist, _ = _device_beam(m, statics, [3, -1], k, G, 0.0, True, True, out_size=1)
        _, ref, _ = _device_beam(m, statics, [3, -1], B, 1, 0.0, True, True, out_size=1)
        for g in range(G):
            s = slice(g * B, (g + 1) * B)
            par = hist[0][:, :, s].clone()
            par[1:] -= g * B                  # slots of group g at t > 0; every t = 0 pick has the BOS row 0 as parent
            mine = [par, hist[1][:, :, s], hist[2][:, :, s], hist[3][:, :, s]]
            diff = torch.zeros(ref[0].shape[:2], dtype=torch.bool, device=ref[0].device)     # (T, b)
            for x, y in zip(mine, ref):
                diff |= (x != y).any(2)
            for c in diff.any(0).nonzero().flatten().tolist():
                t = int(diff[:, c].nonzero()[0])
                sl = [x[t, c].cpu() for x in mine], [y[t, c].cpu() for y in ref]
                (pp, pw, pg, ps), (rp, rw, rg, rs) = sl
                j = int(((pp != rp) | (pw != rw) | (pg != rg) | (ps != rs)).nonzero()[0])      # first slot that differs
                assert pp[j] == rp[j] and pg[j] == rg[j] and ps[j] == rs[j] and pw[j] < rw[j], (k, G, g, c, t, sl)
                tied.add(c)
        print("captions with a rounding tie", k, G, len(tied))
        assert len(tied) <= captions // 20, (k, G, sorted(tied))        # rare: the rest matched bit for bit


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
def test_one_group_is_unchanged():
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"], fx["verbs_gt"])
    eng = m._engine()
    calls = [(lambda **kw: m.beam_search_v(dev, [3, -1], 4, 2, gt=True, **kw), 2),
             (lambda **kw: m.beam_search(dev[:2], [3, 1], 6, 6, **kw), 3)]
    for call, G in calls:
        base = []
        # eager, graph capture, replay, replay: a penalty with one group changes nothing, not even the graph key
        for kw in (dict(), dict(num_beam_groups=1), dict(), dict(num_beam_groups=1, diversity_penalty=3.5)):
            l0 = eng.launch_count()
            res = _flat(call(**kw))
            torch.cuda.synchronize()
            base.append((res, eng.launch_count() - l0))
        for res, launches in base[1:]:
            assert launches == base[0][1]
            assert all(torch.equal(x, y) for x, y in zip(res, base[0][0]))
        on = _flat(call(num_beam_groups=G, diversity_penalty=2.0))
        assert eng.beam_diversity == (1, 0.0)
        assert any(not torch.equal(x, y) for x, y in zip(on, base[0][0]))
        for _ in range(3):                                           # off again: the old graph replays
            l0 = eng.launch_count()
            res = _flat(call())
            torch.cuda.synchronize()
            assert eng.launch_count() - l0 == base[0][1]
            assert all(torch.equal(x, y) for x, y in zip(res, base[0][0]))


# ----------------------------------------------------------------------------- both head paths
@pytest.mark.gpu
def test_trace_path_selects_what_the_fused_head_selects():
    """trace_steps runs k_softmax_topk over the full rows; the default runs the fused k_vocab_merge head."""
    fx, m = _small_a()
    for statics, use_verbs, gt in (((fx["det"], fx["det_seqs"]), False, False),
                                   ((fx["det"], fx["det_seqs"], fx["verbs_gt"]), True, True)):
        for k, G, lam in ((6, 3, 1.0), (4, 2, 0.5)):
            df, hf, _ = _device_beam(m, statics, [3, -1], k, G, lam, use_verbs, gt, trace=False)
            dt, ht, extra = _device_beam(m, statics, [3, -1], k, G, lam, use_verbs, gt, trace=True)
            for x, y in zip(hf[:3], ht[:3]):
                assert torch.equal(x, y)
            assert torch.equal(df[0], dt[0]) and torch.equal(df[1], dt[1])
            assert bool(torch.isfinite(extra["step_out"]).all())


# ----------------------------------------------------------------------------- independence
@pytest.mark.gpu
def test_stacked_decode_equals_its_parts_and_pipeline():
    """1000 captions in one decode equal ten 100-caption decodes bit for bit; DecodePipeline with the keywords equals
    direct calls."""
    from gpu_common import make_model
    from vsrdec import DecodePipeline
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    W["out_fc.weight"] = W["out_fc.weight"] * 100.0
    m = make_model(d, W)
    parts = _config2_parts(10)
    big = tuple(torch.cat([p[i] for p in parts]) for i in range(3))
    kw = dict(gt=True, num_beam_groups=3, diversity_penalty=1.0)
    ref = [m.beam_search_v(_cuda(*p), [3, -1], 6, 1, **kw) for p in parts]
    (wb, gb), (lwb, lgb) = m.beam_search_v(_cuda(*big), [3, -1], 6, 1, **kw)
    for i, ((w, g), (lw, lg)) in enumerate(ref):
        s = slice(100 * i, 100 * (i + 1))
        assert torch.equal(w, wb[s]) and torch.equal(g, gb[s]) and torch.equal(lw, lwb[s]) and torch.equal(lg, lgb[s]), i
    (w0, _), _ = m.beam_search_v(_cuda(*parts[0]), [3, -1], 6, 1, gt=True)
    assert not torch.equal(w0, ref[0][0][0])
    pipe = DecodePipeline([m], [3, -1], 6, 1, gt=True, stack=2, num_beam_groups=3, diversity_penalty=1.0)
    host = [tuple(t.pin_memory() for t in p) for p in parts[:4]]
    for i, (w, g, lw, lg) in enumerate(pipe.run(host)):
        assert torch.equal(w, ref[i][0][0].cpu()) and torch.equal(lw, ref[i][1][0].cpu()), i


@pytest.mark.gpu
def test_ffma_twin_subprocess():
    """VSRDEC_GEMM=simt (k_softmax_topk on every step): the diverse beam search passes the oracle check too."""
    code = ("import sys; sys.path[:0] = ['tests', '.', 'vsr-guided-cic_b200']\n"
            "import test_gpu_diverse_beam as M\n"
            "from common import load_golden\n"
            "from gpu_common import make_model\n"
            "fx = load_golden('small_a.pt'); d, W = fx['dims_obj'], fx['weights']\n"
            "m = make_model(d, W, fx['verb_table'])\n"
            "assert m._engine().gemm_kind() == 'simt-fp32'\n"
            "st = (fx['det'], fx['det_seqs'], fx['verbs_tab'])\n"
            "s = M._check('simt', W, d, st, [3, -1], 6, 3, 2.0, m, True, False, fx['verb_table'])\n"
            "assert s['changed'] > 0\n"
            "print('simt ok')\n")
    env = dict(os.environ, VSRDEC_GEMM="simt")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "simt ok" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# ----------------------------------------------------------------------------- errors
@pytest.mark.gpu
def test_invalid_arguments_raise_before_anything_runs():
    from vsrdec import VsrError
    from vsrdec._lib import c_i64
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"], fx["verbs_gt"])
    m.beam_search(dev[:2], [3, -1], 4)
    eng = m._engine()
    torch.cuda.synchronize()
    l0 = eng.launch_count()
    bad = [dict(num_beam_groups=g) for g in (0, 9, -1, True, 2.0, "2", None)]
    bad += [dict(num_beam_groups=2, diversity_penalty=p) for p in (-1.0, float("inf"), float("nan"), 1e39, True, "1",
                                                                   None)]
    bad += [dict(num_beam_groups=3, diversity_penalty=1.0)]             # 3 does not divide beam 4
    for kw in bad:
        for call in (lambda: m.beam_search(dev[:2], [3, -1], 4, **kw),
                     lambda: m.beam_search_v(dev, [3, -1], 4, gt=True, **kw)):
            with pytest.raises(VsrError):
                call()
    for g, p in ((0, 0.0), (9, 0.0), (True, 1.0), (2, -0.5), (2, float("nan")), (2, True), (2, "1")):
        with pytest.raises(VsrError):
            eng.set_beam_diversity(g, p)
    assert eng.launch_count() == l0 and eng.beam_diversity == (1, 0.0)
    h = eng.handle
    for g, p in ((0, 0.0), (9, 0.0), (2, -1.0), (2, float("nan")), (2, float("inf"))):
        assert eng.lib.vsr_set_beam_diversity(h, g, p) == -1
    assert eng.lib.vsr_set_beam_diversity(h, 3, 0.5) == 0
    out = [torch.empty((fx["det"].size(0), 1, fx["dims_obj"].seq_len), device=DEV, dtype=dt)
           for dt in (torch.long, torch.long, torch.float32, torch.float32)]
    eos = (c_i64 * 2)(3, -1)
    assert eng.lib.vsr_beam_search(h, 4, 1, eos, 0, 0, *[x.data_ptr() for x in out], None, None) == -1
    torch.cuda.synchronize()
    assert eng.launch_count() == l0
    assert eng.lib.vsr_beam_search(h, 6, 1, eos, 0, 0, *[x.data_ptr() for x in out], None, None) == 0
    assert eng.lib.vsr_set_beam_diversity(h, 1, 0.0) == 0
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- CPU-only
def _row(V, cur, vals):
    """A candidate score tensor (cur * V * 2) at -50 with vals {(j, w, gate): score}."""
    f = torch.full((cur, V, 2), -50.0)
    for (j, w, g), v in vals.items():
        f[j, w, g] = v
    return f.flatten()


def _fi(V, j, w, g):
    return j * 2 * V + w * 2 + g


def test_select_groups_restatement():
    V = 10
    # t = 0: every group expands the BOS row; with lambda = 0 they pick the same candidates
    f = _row(V, 1, {(0, 3, 0): -1.0, (0, 4, 0): -1.5, (0, 5, 1): -2.0})
    live, frc = [True], [False]
    assert select_groups(f, 1, 4, 2, 0.0, live, frc) == [_fi(V, 0, 3, 0), _fi(V, 0, 4, 0)] * 2
    # lambda = 1: group 1 sees words 3 and 4 at keys -2.0 / -2.5 and word 5 at -2.0; the tie of words 3 and 5 goes to
    # the lower flat index (6 before 11)
    assert select_groups(f, 1, 4, 2, 1.0, live, frc) == [_fi(V, 0, 3, 0), _fi(V, 0, 4, 0),
                                                         _fi(V, 0, 3, 0), _fi(V, 0, 5, 1)]
    # both gates of a word carry the word's count
    f = _row(V, 1, {(0, 3, 0): -1.0, (0, 3, 1): -1.1, (0, 6, 0): -1.6})
    assert select_groups(f, 1, 2, 2, 1.0, live, frc) == [_fi(V, 0, 3, 0), _fi(V, 0, 6, 0)]
    assert select_groups(f, 1, 2, 2, 0.0, live, frc) == [_fi(V, 0, 3, 0), _fi(V, 0, 3, 0)]
    # t > 0, k = 4, G = 2: group 1 only sees parents 2 and 3
    f = _row(V, 4, {(0, 1, 0): -1.0, (1, 2, 0): -1.2, (2, 1, 0): -1.1, (3, 7, 0): -3.0, (2, 8, 1): -2.9})
    live, frc = [True] * 4, [False] * 4
    assert select_groups(f, 4, 4, 2, 0.0, live, frc) == [_fi(V, 0, 1, 0), _fi(V, 1, 2, 0),
                                                         _fi(V, 2, 1, 0), _fi(V, 2, 8, 1)]
    assert select_groups(f, 4, 4, 2, 2.5, live, frc) == [_fi(V, 0, 1, 0), _fi(V, 1, 2, 0),
                                                         _fi(V, 2, 8, 1), _fi(V, 3, 7, 0)]
    # a verb-forced row of group 1 is never penalised ...
    assert select_groups(f, 4, 4, 2, 2.5, live, [False, False, True, False])[2:] == [_fi(V, 2, 1, 0), _fi(V, 2, 8, 1)]
    # ... and a forced row's pick still counts against later groups
    assert select_groups(f, 4, 4, 2, 2.5, live, [True, False, False, False])[2:] == [_fi(V, 2, 8, 1), _fi(V, 3, 7, 0)]
    # a frozen parent's pick does not count, and a frozen row's candidates are never penalised
    assert select_groups(f, 4, 4, 2, 2.5, [False, True, True, True], frc)[2:] == [_fi(V, 2, 1, 0), _fi(V, 2, 8, 1)]
    assert select_groups(f, 4, 4, 2, 2.5, [True, True, False, True], frc)[2:] == [_fi(V, 2, 1, 0), _fi(V, 2, 8, 1)]
    # G = k: one beam per group, each group penalised by all earlier picks; a small penalty lets word 1 come back
    f = _row(V, 1, {(0, 1, 0): -1.0, (0, 2, 0): -1.4, (0, 3, 0): -1.9})
    assert select_groups(f, 1, 3, 3, 1.0, [True], [False]) == [_fi(V, 0, 1, 0), _fi(V, 0, 2, 0), _fi(V, 0, 3, 0)]
    assert select_groups(f, 1, 3, 3, 0.5, [True], [False]) == [_fi(V, 0, 1, 0), _fi(V, 0, 2, 0), _fi(V, 0, 1, 0)]


def test_group_keys_are_float32_rounded():
    V = 4
    f = _row(V, 1, {(0, 1, 0): -1.0})
    _, key = group_keys(f, 1, V, 1, 1, 0.1, [True], [False], [_fi(V, 0, 1, 0)] * 3)
    lam = torch.tensor(0.1, dtype=torch.float32)
    assert key.dtype == torch.float32 and float(key[0, 1, 0]) == float(torch.tensor(-1.0) - lam * 3)


def test_argument_check_without_a_device():
    from vsrdec import VsrError
    from vsrdec.engine import check_beam_diversity
    check_beam_diversity(1, 0.0)
    check_beam_diversity(1, 5.0, 7)                  # one group divides any beam
    check_beam_diversity(3, 0, 6)
    check_beam_diversity(8, 2.5, 8)
    check_beam_diversity(2, 1e30)
    for args in ((0, 0.0), (9, 0.0), (True, 0.0), (2.0, 0.0), ("2", 0.0), (None, 0.0), (2, -1.0), (2, float("inf")),
                 (2, float("nan")), (2, 1e39), (2, True), (2, "1"), (2, None), (3, 1.0, 4), (2, 0.0, 5)):
        with pytest.raises(VsrError):
            check_beam_diversity(*args)


def test_signatures_and_binding():
    import inspect
    import re
    from models.CaptioningModel import CaptioningModel
    from vsrdec import DecodePipeline, EvalFlow, EXPORTED_SYMBOLS
    for fn in (CaptioningModel.beam_search, CaptioningModel.beam_search_v, CaptioningModel.beam_search_v_indexed,
               DecodePipeline.__init__, EvalFlow.__init__):
        ps = inspect.signature(fn).parameters
        assert ps["num_beam_groups"].default == 1 and ps["diversity_penalty"].default == 0.0, fn
    assert "vsr_set_beam_diversity" in EXPORTED_SYMBOLS
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "vsrdec.h")).read(), flags=re.S)
    assert re.search(r"int vsr_set_beam_diversity\(vsr_handle h, int32_t groups, float penalty\);", src)


def test_model_rejects_bad_settings_before_the_engine():
    """The drivers validate the keywords before they touch the engine (here: a CPU model, whose engine would raise a
    different error)."""
    from vsrdec import VsrError
    from models import ControllableCaptioningModel
    m = ControllableCaptioningModel(8, 10, 2, det_feat_size=8, input_encoding_size=4, rnn_size=4, att_size=4,
                                    verb_tables=({}, {}))
    det, ds = torch.zeros(2, 3, 8), torch.zeros(2, 4, 2, 8)
    verbs = torch.zeros(2, 4)
    for call in (lambda: m.beam_search((det, ds), [3, -1], 4, num_beam_groups=3),
                 lambda: m.beam_search_v((det, ds, verbs), [3, -1], 4, num_beam_groups=2, diversity_penalty=-1.0),
                 lambda: m.beam_search_v_indexed((det, torch.zeros(2, 4, 2, dtype=torch.int32), verbs), [3, -1], 4,
                                                 num_beam_groups=0)):
        with pytest.raises(VsrError, match="num_beam_groups|diversity_penalty"):
            call()


def test_evalflow_passes_the_keywords():
    from vsrdec import EvalFlow

    class Recorder:
        def beam_search_v_indexed(self, statics, eos, beam_size, out_size, **kw):
            self.kw = kw
            return "decoded"

    rec = Recorder()
    flow = EvalFlow(rec, None, [3, -1], beam_size=6, num_beam_groups=3, diversity_penalty=1.5)
    b = {"detections": torch.zeros(2, 3, 8), "slot_index": torch.zeros(2, 4, 2, dtype=torch.int32)}
    assert flow._decode(b, torch.arange(4).expand(2, 4), torch.zeros(2, 4)) == "decoded"
    assert rec.kw["num_beam_groups"] == 3 and rec.kw["diversity_penalty"] == 1.5
