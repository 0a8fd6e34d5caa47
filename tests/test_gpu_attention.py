"""Per-word attention of the decode drivers (vsr_set_attention_capture / vsr_get_attention, return_attention=True).

The reference computes `alpha` inside step_v (controllable_captioning.py:159-169) and never returns it.  The oracle's
decoder_step is kept as the reference pins it, so the reference attention here is a restatement of its first half
(`oracle_step_attention`, the same torch CPU ops in the same order), checked against decoder_step's own state outputs.
During a replay through the oracle's drivers, `recording_attention` records it for every step.

GPU tests are marked one by one: the CPU-only cases at the end run without a device."""
import contextlib
import os
import re
import subprocess

import pytest
import torch
import torch.nn.functional as F

from common import load_golden, verify_device_beam
from oracle import vsr_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
ALPHA_ATOL = 1e-4      # device vs oracle attention weights (the max error measured per config is printed)


def _cuda(*ts):
    return tuple(t.to(DEV) for t in ts)


# ----------------------------------------------------------------------------- reference attention
def oracle_step_attention(W, d, t, state, prev_outputs, statics, seqs, mode):
    """alpha (N, R+1) and slot pointer (N) of one O.decoder_step call with these arguments, plus the (h1, c1) it
    produces: decoder_step's lines up to the renormalised alpha (vsr_oracle.py, controllable_captioning.py:126-169)."""
    det = statics[0]
    n = det.size(0)
    det_mask = (torch.sum(det, -1, keepdim=True) != 0).to(det.dtype)
    img = torch.sum(det, 1) / torch.sum(det_mask, 1)
    (h1, c1), (h2, c2), ptr = state
    if mode == "teacher_forcing":
        word_in = seqs[0][:, t]
        det_curr = seqs[1][:, t]
        ptr = torch.full((n,), t, dtype=torch.long)
    else:
        if t == 0:
            word_in = torch.full((n,), d.bos_idx, dtype=torch.long)
        else:
            word_in = prev_outputs[0]
            ptr = torch.clamp(ptr + prev_outputs[1], 0, statics[1].shape[1] - 1)
        det_curr = statics[1][torch.arange(n), ptr]
    xt = F.embedding(word_in, W["embed.weight"])
    in1 = torch.cat([h2, img, xt], 1) if d.h2_first_lstm else torch.cat([img, xt], 1)
    s_gate = torch.sigmoid(F.linear(in1, W["W1_is.weight"], W["W1_is.bias"])
                           + F.linear(h1, W["W1_hs.weight"], W["W1_hs.bias"]))
    h1, c1 = O._lstm_cell(in1, h1, c1, W["lstm_cell_1.weight_ih"], W["lstm_cell_1.weight_hh"],
                          W["lstm_cell_1.bias_ih"], W["lstm_cell_1.bias_hh"])
    s_t = s_gate * torch.tanh(c1)
    sentinel = F.linear(s_t, W["s_fc.weight"], W["s_fc.bias"]).unsqueeze(1)
    regions = torch.cat([sentinel, det_curr], 1)
    regions_mask = (torch.sum(regions, -1, keepdim=True) != 0).to(det.dtype)
    ha = F.linear(h1, W["att_ha.weight"])
    det_w = F.linear(torch.tanh(F.linear(det_curr, W["att_va.weight"]) + ha.unsqueeze(1)), W["att_a.weight"])
    sent_w = F.linear(torch.tanh(F.linear(s_t, W["att_sa.weight"]) + ha).unsqueeze(1), W["att_s.weight"])
    alpha = F.softmax(torch.cat([sent_w, det_w], 1), 1)
    alpha = regions_mask * alpha
    alpha = alpha / torch.sum(alpha, 1, keepdim=True)
    return alpha.squeeze(-1), ptr, (h1, c1)


@contextlib.contextmanager
def recording_attention():
    """While active, every O.decoder_step call (also those made by O.beam_search / O.forward_teacher) appends
    (alpha (N, R+1), slot (N)) of that step to the yielded list; decoder_step's outputs are untouched."""
    rec = []
    orig = O.decoder_step

    def step(W, d, t, state, prev_outputs, statics, seqs, mode, use_verbs=False, gt=False, verb_table=None):
        alpha, ptr, _ = oracle_step_attention(W, d, t, state, prev_outputs, statics, seqs, mode)
        rec.append((alpha, ptr))
        return orig(W, d, t, state, prev_outputs, statics, seqs, mode, use_verbs=use_verbs, gt=gt, verb_table=verb_table)

    O.decoder_step = step
    try:
        yield rec
    finally:
        O.decoder_step = orig


def beam_path(hist, out_size):
    """Rows of every step along each returned beam's back-pointer path, (b, out_size, T), from the device history:
    final order = stable descending sort of the last step's scores, row of step t = caption * cur_t + parent slot.
    Also returns the words and gates along the path (must equal the returned tokens)."""
    parent, word, gate, score = [x.cpu().long() for x in hist[:3]] + [hist[3].cpu()]
    T, b, k = parent.shape
    slot = torch.sort(score[T - 1], dim=1, descending=True, stable=True).indices[:, :out_size]
    rows = torch.empty((b, out_size, T), dtype=torch.long)
    words, gates = torch.empty_like(rows), torch.empty_like(rows)
    cap = torch.arange(b).unsqueeze(1)
    for t in range(T - 1, -1, -1):
        words[:, :, t] = torch.gather(word[t], 1, slot)
        gates[:, :, t] = torch.gather(gate[t], 1, slot)
        slot = torch.gather(parent[t], 1, slot)
        rows[:, :, t] = cap * (1 if t == 0 else k) + slot
    return rows, words, gates


def check_structure(att, gates, det_seqs, tag):
    """Rows sum to 1, exact zeros at padding regions, slot recursion from the returned gates.  att/gates (..., T)."""
    alpha, slot = att["alpha"].cpu(), att["slot"].cpu()
    gates = gates.cpu()
    L = det_seqs.size(1)
    assert alpha.shape[:-1] == slot.shape == gates.shape, tag
    assert (alpha >= 0).all(), tag
    assert float((alpha.double().sum(-1) - 1).abs().max()) <= 1e-6, tag
    assert (slot[..., 0] == 0).all(), tag
    assert torch.equal(slot[..., 1:], torch.clamp(slot[..., :-1] + gates[..., :-1], 0, L - 1)), tag
    b = det_seqs.size(0)
    pad_regions = det_seqs.sum(-1) == 0                                      # (b, L, R)
    pad = pad_regions[torch.arange(b).unsqueeze(1), slot.reshape(b, -1)].reshape(alpha.shape[:-1] + (alpha.size(-1) - 1,))
    assert (alpha[..., 1:][pad] == 0).all(), f"{tag}: nonzero weight on a padding region"


def compare_beam(att, rec, rows, tag):
    """Device attention along the path vs the oracle's recorded rows; slot exact, alpha within ALPHA_ATOL."""
    alpha, slot = att["alpha"].cpu(), att["slot"].cpu()
    T = rows.size(-1)
    assert len(rec) == T
    err = 0.0
    for t in range(T):
        ra, rp = rec[t]
        r = rows[..., t]
        assert torch.equal(slot[..., t], rp[r]), f"{tag}: slot differs at t={t}"
        err = max(err, float((alpha[..., t, :] - ra[r]).abs().max()))
    print(f"ATTENTION {tag}: max |alpha - oracle| = {err:.3e}")
    assert err <= ALPHA_ATOL, f"{tag}: alpha error {err:.3e}"
    return err


def _full_model(d, seed, sharpen=None, table=None):
    from gpu_common import make_model
    W = O.init_weights(d, seed=seed)
    if sharpen:
        W["out_fc.weight"] = W["out_fc.weight"] * sharpen
    return W, make_model(d, W, table)


def _config2_inputs(b=100, seed=1002):
    return O.synth_inputs(b, 50, 10, 20, 2048, seed=seed, vocab_size=10000, n_det_range=(10, 50), verb_slots=(2,),
                          verb_vocab_id=17)


# ----------------------------------------------------------------------------- 1. capture changes nothing
@pytest.mark.gpu
def test_capture_changes_no_output_and_replays_from_the_graph():
    """Config 2 raw (the benchmarked workload): capture off, on, on again (graph replay).  Tokens, log-probs and the
    history are bit-identical across the three; the attention of the two captured calls too; capture off launches
    exactly what it did before capture existed on the handle."""
    from vsrdec import VsrError
    d = O.Dims()
    W, m = _full_model(d, 1234)
    det, ds, verbs = _config2_inputs()
    dev = _cuda(det, ds, verbs)
    m.beam_search_v(dev, [3, -1], 5, 1, gt=True)            # warm: first sighting of the capture-off key
    eng = m._eng
    runs = []
    for ret in (False, True, True):
        l0 = eng.launch_count()
        res = m.beam_search_v(dev, [3, -1], 5, 1, gt=True, return_attention=ret)
        hist = eng.history()
        torch.cuda.synchronize()
        runs.append((res, [h.clone() for h in hist], eng.launch_count() - l0))
    (o0, lp0), h0, n0 = runs[0]
    for (res, h, n) in runs[1:]:
        assert torch.equal(res[0][0], o0[0]) and torch.equal(res[0][1], o0[1])
        assert torch.equal(res[1][0], lp0[0]) and torch.equal(res[1][1], lp0[1])
        assert all(torch.equal(a, b) for a, b in zip(h, h0))
        assert n == n0 + 1                                  # the decode's launches plus the gather of the attention
    a1, a2 = runs[1][0][2], runs[2][0][2]
    assert a1["alpha"].shape == (100, d.seq_len, 21) and a1["slot"].shape == (100, d.seq_len)
    assert a1["alpha"].dtype == torch.float32 and a1["slot"].dtype == torch.int64
    assert torch.equal(a1["alpha"], a2["alpha"]) and torch.equal(a1["slot"], a2["slot"])
    check_structure(a1, o0[1], ds, "config2 raw")
    # capture is off again after a return_attention call: a plain decode launches as before and has no attention
    l0 = eng.launch_count()
    m.beam_search_v(dev, [3, -1], 5, 1, gt=True)
    assert eng.launch_count() - l0 == n0
    with pytest.raises(VsrError):
        eng.attention()


# ----------------------------------------------------------------------------- 2./3. beam search vs the oracle
BEAM_CONFIGS = {
    "config2_raw": dict(cfg=2, sharpen=None),
    "config2_x100": dict(cfg=2, sharpen=100.0),
    "config3_det": dict(cfg=3, sharpen=None),
    "config4_flickr": dict(cfg=4, sharpen=None),
    "serial_R40": dict(cfg=0, sharpen=30.0),
}


def _beam_config(cfg, sharpen):
    table = None
    if cfg == 2:
        d = O.Dims()
        statics, k, gt, seed = _config2_inputs(), 5, True, 1234
    elif cfg == 3:
        d = O.Dims()
        table = O.synth_verb_table(2662, d.vocab_size, seed=11)
        statics = O.synth_inputs(100, 100, 10, 20, 2048, seed=1003, vocab_size=d.vocab_size, n_det_range=(10, 100),
                                 verb_slots=(1, 3), verb_id_range=(0, 2700))
        k, gt, seed = 5, False, 1234
    elif cfg == 4:
        d = O.Dims(vocab_size=7000)
        statics = O.synth_inputs(100, 100, 10, 20, 2048, seed=1004, vocab_size=d.vocab_size, n_det_range=(10, 100),
                                 verb_slots=(2,), verb_vocab_id=23, one_region_slots=True)
        k, gt, seed = 5, True, 4242
    else:       # R + 1 > 32: the serial softmax branch of the attention kernel
        d = O.Dims(seq_len=10, vocab_size=300, det_feat_size=128, input_encoding_size=32, rnn_size=64, att_size=32)
        statics = O.synth_inputs(12, 60, 6, 40, 128, seed=31, vocab_size=d.vocab_size, n_det_range=(20, 60),
                                 real_slots=(3, 6), verb_slots=(1,), verb_vocab_id=11)
        k, gt, seed = 4, True, 5
    W, m = _full_model(d, seed, sharpen, table)
    return d, W, m, statics, k, gt, table


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(BEAM_CONFIGS))
def test_beam_attention_matches_oracle_along_the_path(name):
    """Every returned beam (out_size = beam) at every step: the device's alpha and slot against the oracle's row at
    the beam's back-pointer path, with the device trajectory replayed through the oracle (as verify_device_beam)."""
    d, W, m, statics, k, gt, table = _beam_config(**BEAM_CONFIGS[name])
    (w, g), (lw, lg), att = m.beam_search_v(_cuda(*statics), [3, -1], k, k, gt=gt, return_attention=True)
    hist = m._eng.history()
    torch.cuda.synchronize()
    R = statics[1].size(2)
    assert att["alpha"].shape == (statics[0].size(0), k, d.seq_len, R + 1)
    rows, pw, pg = beam_path(hist, k)
    assert torch.equal(pw, w.cpu()) and torch.equal(pg, g.cpu())
    with recording_attention() as rec:
        v, _, _ = verify_device_beam(W, d, statics, [3, -1], k, hist, True, gt, table)
    assert not v.violations, v.violations[:5]
    compare_beam(att, rec, rows, name)
    check_structure(att, g, statics[1], name)


# ----------------------------------------------------------------------------- 4. caption independence
@pytest.mark.gpu
def test_attention_is_independent_of_the_batch():
    """A caption's attention is bit-identical decoded alone, in the 100-caption batch and in a 230-caption (1150-row,
    CTA-pair GEMM kernels) stacked decode."""
    d = O.Dims()
    W, m = _full_model(d, 1234)
    a = _config2_inputs()
    extra = _config2_inputs(130, seed=1003)
    stacked = tuple(torch.cat([x, y], 0) for x, y in zip(a, extra))
    _, _, att100 = m.beam_search_v(_cuda(*a), [3, -1], 5, 1, gt=True, return_attention=True)
    _, _, att230 = m.beam_search_v(_cuda(*stacked), [3, -1], 5, 1, gt=True, return_attention=True)
    for c in (0, 37, 99):
        _, _, att1 = m.beam_search_v(_cuda(*(x[c:c + 1] for x in a)), [3, -1], 5, 1, gt=True, return_attention=True)
        for key in ("alpha", "slot"):
            assert torch.equal(att1[key][0], att100[key][c]), (c, key)
            assert torch.equal(att230[key][c], att100[key][c]), (c, key)


# ----------------------------------------------------------------------------- 5. index form
@pytest.mark.gpu
@pytest.mark.parametrize("shared_image", [False, True])
def test_indexed_attention_and_detection_rows(shared_image):
    d = O.Dims()
    W, m = _full_model(d, 1234, 100.0)
    det, idx, verbs = O.synth_inputs_indexed(24, 50, 10, 20, 2048, seed=1006, n_det_range=(10, 50))
    if shared_image:
        det = det[:1].expand(24, 50, 2048)
        idx = idx.clamp(max=int((det[0].sum(-1) != 0).sum()) - 1)
    ds = O.materialize_slots(det, idx)
    dev = (det.to(DEV) if not shared_image else det[:1].to(DEV).expand(24, 50, 2048), idx.to(DEV), verbs.to(DEV))
    (w, g), _, att = m.beam_search_v_indexed(dev, [3, -1], 5, 1, gt=True, return_attention=True)
    hist = m._eng.history()
    torch.cuda.synchronize()
    assert att["alpha"].shape == (24, d.seq_len, 21) and att["det_index"].shape == (24, d.seq_len, 20)
    assert att["det_index"].dtype == torch.int64
    slot = att["slot"].cpu()
    assert torch.equal(att["det_index"].cpu(), idx.long()[torch.arange(24).unsqueeze(1), slot])
    rows, pw, _ = beam_path(hist, 1)
    assert torch.equal(pw[:, 0], w.cpu())
    with recording_attention() as rec:
        v, _, _ = verify_device_beam(W, d, (det.contiguous(), ds, verbs), [3, -1], 5, hist, True, True)
    assert not v.violations, v.violations[:5]
    compare_beam({k: x.unsqueeze(1) for k, x in att.items()}, rec, rows, f"indexed shared_image={shared_image}")
    check_structure(att, g, ds, "indexed")


# ----------------------------------------------------------------------------- 6. the other drivers
@pytest.mark.gpu
def test_forward_attention_matches_teacher_forced_oracle():
    """Config 5 (teacher forcing, B=100, T=20): slot == t and alpha against the oracle's teacher-forced unroll."""
    d = O.Dims()
    W, m = _full_model(d, 1234)
    det, ds, _ = O.synth_inputs(100, 100, 10, 20, 2048, seed=1005, vocab_size=d.vocab_size, n_det_range=(10, 100))
    caps = torch.randint(0, d.vocab_size, (100, 20), generator=torch.Generator().manual_seed(7))
    ctrl = torch.stack([ds[:, min(t // 2, 9)] for t in range(20)], 1).contiguous()
    out, gate = m((det.to(DEV),), (caps.to(DEV), ctrl.to(DEV)))
    out2, gate2, att = m((det.to(DEV),), (caps.to(DEV), ctrl.to(DEV)), return_attention=True)
    torch.cuda.synchronize()
    assert torch.equal(out, out2) and torch.equal(gate, gate2)
    assert att["alpha"].shape == (100, 20, 21)
    assert torch.equal(att["slot"].cpu(), torch.arange(20).expand(100, 20))
    with recording_attention() as rec, torch.no_grad():
        O.forward_teacher(W, d, (det,), (caps, ctrl))
    rows = torch.arange(100).view(100, 1, 1).expand(100, 1, 20)
    compare_beam({k: x.unsqueeze(1) for k, x in att.items()}, rec, rows, "config5 forward")
    alpha = att["alpha"].cpu()
    assert float((alpha.double().sum(-1) - 1).abs().max()) <= 1e-6
    assert (alpha[..., 1:][ctrl.sum(-1) == 0] == 0).all()


def _replay_rows(W, d, statics, words, gates):
    """The oracle fed the device's own words and gates (feedback mode), recording its attention."""
    b = statics[0].size(0)
    state, prev = O.init_state(d, b), None
    with recording_attention() as rec, torch.no_grad():
        for t in range(d.seq_len):
            _, state = O.decoder_step(W, d, t, state, prev, statics, None, "feedback")
            prev = (words[:, t], gates[:, t])
    return rec


@pytest.mark.gpu
def test_greedy_and_sampling_attention_match_oracle_replay():
    from gpu_common import make_model
    fx = load_golden("small_a.pt")
    d, W = fx["dims_obj"], fx["weights"]
    m = make_model(d, W, fx["verb_table"])
    det, ds = fx["det"], fx["det_seqs"]
    b = det.size(0)
    rows = torch.arange(b).view(b, 1, 1).expand(b, 1, d.seq_len)
    w0, g0 = m.test(*_cuda(det, ds))
    w, g, att = m.test(*_cuda(det, ds), return_attention=True)
    assert torch.equal(w, w0) and torch.equal(g, g0)
    rec = _replay_rows(W, d, (det, ds), w.cpu(), g.cpu())
    compare_beam({k: x.unsqueeze(1) for k, x in att.items()}, rec, rows, "greedy")
    check_structure(att, g, ds, "greedy")
    (sw0, sg0), (lw0, lg0) = m.sample_rl(*_cuda(det, ds), seed=123)
    (sw, sg), (lw, lg), satt = m.sample_rl(*_cuda(det, ds), seed=123, return_attention=True)
    assert torch.equal(sw, sw0) and torch.equal(sg, sg0) and torch.equal(lw, lw0) and torch.equal(lg, lg0)
    _, _, satt2 = m.sample_rl(*_cuda(det, ds), seed=123, return_attention=True)
    assert torch.equal(satt["alpha"], satt2["alpha"]) and torch.equal(satt["slot"], satt2["slot"])
    rec = _replay_rows(W, d, (det, ds), sw.cpu(), sg.cpu())
    compare_beam({k: x.unsqueeze(1) for k, x in satt.items()}, rec, rows, "sample_rl")
    check_structure(satt, sg, ds, "sample_rl")


# ----------------------------------------------------------------------------- 7. errors
@pytest.mark.gpu
def test_get_attention_after_a_decode_without_capture_is_a_state_error():
    import ctypes
    from gpu_common import make_model
    from vsrdec import VsrError
    fx = load_golden("small_a.pt")
    m = make_model(fx["dims_obj"], fx["weights"], fx["verb_table"])
    dev = _cuda(fx["det"], fx["det_seqs"], fx["verbs_gt"])
    m.beam_search_v(dev, [3, -1], 3, 1, gt=True, return_attention=True)
    m.beam_search_v(dev, [3, -1], 3, 1, gt=True)
    with pytest.raises(VsrError, match="without attention capture"):
        m._eng.attention()
    buf = torch.empty(1 << 16, device=DEV)
    assert m._eng.lib.vsr_get_attention(m._eng.handle, buf.data_ptr(), buf.data_ptr(), None) == -4    # VSR_ESTATE
    m.test(*dev[:2])
    with pytest.raises(VsrError):
        m._eng.attention()


# ----------------------------------------------------------------------------- 8. CPU-only
def test_oracle_step_attention_follows_decoder_step():
    """The reference attention starts from decoder_step's own inputs: its (h1, c1, slot) equal decoder_step's outputs
    bit for bit; its rows sum to 1 and are 0 at padding regions; recording leaves decoder_step's outputs bit-identical."""
    d = O.Dims(seq_len=6, vocab_size=97, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    W = O.init_weights(d, seed=5)
    det, ds, verbs = O.synth_inputs(5, 9, 5, 6, d.det_feat_size, seed=21, vocab_size=d.vocab_size, n_det_range=(3, 9),
                                    real_slots=(2, 5), verb_slots=(1,), verb_vocab_id=11)
    g = torch.Generator().manual_seed(3)
    state, prev = O.init_state(d, 5), None
    with torch.no_grad():
        for t in range(d.seq_len):
            alpha, ptr, (h1, c1) = oracle_step_attention(W, d, t, state, prev, (det, ds, verbs), None, "feedback")
            (out, gate), new = O.decoder_step(W, d, t, state, prev, (det, ds, verbs), None, "feedback", use_verbs=True,
                                              gt=True)
            with recording_attention() as rec:
                (out2, gate2), new2 = O.decoder_step(W, d, t, state, prev, (det, ds, verbs), None, "feedback",
                                                     use_verbs=True, gt=True)
            assert torch.equal(out, out2) and torch.equal(gate, gate2)
            assert all(torch.equal(x, y) for x, y in zip(new[0] + new[1] + (new[2],), new2[0] + new2[1] + (new2[2],)))
            assert torch.equal(rec[0][0], alpha) and torch.equal(rec[0][1], ptr)
            assert torch.equal(h1, new[0][0]) and torch.equal(c1, new[0][1]) and torch.equal(ptr, new[2])
            assert alpha.shape == (5, 7)
            assert float((alpha.double().sum(1) - 1).abs().max()) <= 1e-6
            assert (alpha[:, 1:][ds[torch.arange(5), ptr].sum(-1) == 0] == 0).all()
            prev = (torch.randint(0, d.vocab_size, (5,), generator=g), torch.randint(0, 2, (5,), generator=g))
            state = new


def _header_functions():
    src = open(os.path.join(ROOT, "include", "vsrdec.h")).read()
    return set(re.findall(r"\b(vsr_[a-z_0-9]+)\s*\(", re.sub(r"/\*.*?\*/", "", src, flags=re.S)))


def test_header_declares_the_attention_entry_points():
    assert {"vsr_set_attention_capture", "vsr_get_attention"} <= _header_functions()
    import vsrdec
    assert {"vsr_set_attention_capture", "vsr_get_attention"} <= set(vsrdec.EXPORTED_SYMBOLS)


def test_library_exports_the_attention_entry_points():
    import vsrdec
    path = vsrdec.library_path()
    if not os.path.isfile(path):
        pytest.skip("libvsrdec.so is not built")
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (vsr_[a-z_0-9]+)", out))
    assert {"vsr_set_attention_capture", "vsr_get_attention"} <= exported
