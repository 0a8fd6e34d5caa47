"""Sampling decode with several draws per caption, temperature, top-k / top-p truncation and verb forcing
(vsr_sample_ex, DecoderEngine.sample, sample_rl / sample_v).

The reference distribution is `_sets` below: a float64 restatement of the semantics in include/vsrdec.h (temperature,
then top-k, then top-p over the order (x desc, index asc)) applied to the oracle's `decoder_step` rows.  The device's
logits agree with the oracle's to the parity tolerance only, so a word at a set boundary is accepted either way when
its oracle log-prob is within 1e-4 (relative) of the k-th one or when the mass in front of it is within 1e-4 of top_p.

GPU tests are marked one by one: the CPU-only cases at the end run without a device."""
import ctypes
import math
import os
import re
import subprocess

import pytest
import torch

from oracle import vsr_oracle as O
from common import load_golden, rel_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
REL, ABS = 1e-3, 1e-4          # parity tolerance of the returned log-probs
BAND = 1e-4                    # boundary band of the set checks (relative on log-probs, absolute on masses)


def _cuda(*ts):
    return tuple(t.to(DEV) if t is not None else None for t in ts)


def _small_a():
    from gpu_common import make_model
    fx = load_golden("small_a.pt")
    return fx, make_model(fx["dims_obj"], fx["weights"], fx["verb_table"])


def _tol(x):
    return BAND * x.abs() + 1e-5


# ----------------------------------------------------------------------------- float64 reference sets
def _sets(lp, tau=1.0, top_k=0, top_p=1.0):
    """lp (N, V) float64 log-probs of unforced rows.  Returns (probs, allowed, certain), each (N, V):
    probs = the tempered, truncated, renormalised distribution over P; allowed = P widened by the boundary band;
    certain = P narrowed by it (words that are in P whatever the rounding)."""
    lp = lp.double()
    N, V = lp.shape
    k = V if top_k == 0 else min(top_k, V)
    srt, order = torch.sort(-lp, dim=1, stable=True)                 # (x desc, index asc)
    slp = -srt
    pos = torch.arange(V).expand(N, V)
    in_k = pos < k
    z = slp / tau
    e = torch.exp(z - z[:, :1]) * in_k
    q = e / e.sum(1, keepdim=True)
    cum = q.cumsum(1)
    if top_p >= 1.0:
        in_p = in_k
    else:
        m = (cum < top_p).sum(1, keepdim=True).clamp(max=k - 1)      # first entry whose prefix mass reaches top_p
        in_p = pos <= m
    p_sorted = torch.where(in_p, q, torch.zeros_like(q))
    p_sorted = p_sorted / p_sorted.sum(1, keepdim=True)
    probs = torch.zeros_like(lp).scatter_(1, order, p_sorted)
    # mass strictly in front of each word, bounded from below / above over every order the band allows
    cum0 = torch.cat([torch.zeros(N, 1, dtype=lp.dtype), cum], 1)
    neg = (-slp).contiguous()
    lo_cnt = torch.searchsorted(neg, (-(lp + _tol(lp))).contiguous(), right=False)    # entries with lp_u > lp_w + tol
    hi_cnt = torch.searchsorted(neg, (-(lp - _tol(lp))).contiguous(), right=True)     # entries with lp_u >= lp_w - tol
    q_w = torch.zeros_like(lp).scatter_(1, order, q)
    mass_lo = cum0.gather(1, lo_cnt.clamp(max=V))
    mass_hi = cum0.gather(1, hi_cnt.clamp(max=V)) - q_w
    kth = slp[:, k - 1:k]
    allowed = torch.ones_like(lp, dtype=torch.bool)
    certain = torch.zeros_like(lp, dtype=torch.bool).scatter_(1, order, in_p)
    if k < V:
        allowed &= lp >= kth - _tol(kth)
        certain &= lp > kth + _tol(kth)
    if top_p < 1.0:
        allowed &= mass_lo < top_p + BAND
        certain &= mass_hi < top_p - BAND
    return probs, allowed, certain


def _replay(W, d, statics, words, gates, n, use_verbs=False, gt=False, verb_table=None):
    """The oracle along the device's trajectories: rows caption-major (caption * n + draw).  Returns the per-step
    (out, gate) log-probs, float64, (T, N, V) / (T, N, 2)."""
    stat = tuple(s.repeat_interleave(n, 0) if s is not None else None for s in statics)
    N, T = words.shape
    state = O.init_state(d, N)
    prev, outs, gs = None, [], []
    with torch.no_grad():
        for t in range(T):
            (out, gate), state = O.decoder_step(W, d, t, state, prev, stat, None, "feedback", use_verbs, gt, verb_table)
            outs.append(out.double()); gs.append(gate.double())
            prev = (words[:, t], gates[:, t])
    return torch.stack(outs), torch.stack(gs)


def _check_support(W, d, statics, res, n, tau, top_k, top_p, use_verbs=False, gt=False, verb_table=None):
    """Test 3 (and 7): every draw lies in the oracle's P, forced rows take the forced word and gate 1 with log-prob 0,
    and the returned log-probs are the oracle's untempered ones."""
    (w, g), (lw, lg) = res
    T = d.seq_len
    w, g, lw, lg = (x.cpu().reshape(-1, T) for x in (w, g, lw, lg))
    outs, gates = _replay(W, d, statics, w, g, n, use_verbs, gt, verb_table)
    n_forced = 0
    for t in range(T):
        out, gate = outs[t], gates[t]
        forced = (out == 0).sum(1).eq(1) & (out == -1e6).sum(1).eq(out.size(1) - 1)
        n_forced += int(forced.sum())
        free = ~forced
        if forced.any():
            assert torch.equal(w[forced, t], out[forced].argmax(1)), f"step {t}: forced word"
            assert bool((g[forced, t] == 1).all()) and bool((lw[forced, t] == 0).all()) and bool((lg[forced, t] == 0).all())
        if free.any():
            _, allowed, _ = _sets(out[free], tau, top_k, top_p)
            ok = allowed.gather(1, w[free, t:t + 1]).squeeze(1)
            assert bool(ok.all()), f"step {t}: {int((~ok).sum())} draws outside P (tau={tau} k={top_k} p={top_p})"
            assert rel_close(lw[free, t], out[free].gather(1, w[free, t:t + 1]).squeeze(1), REL, ABS)
        assert rel_close(lg[:, t], gate.gather(1, g[:, t:t + 1]).squeeze(1), REL, ABS)
    return n_forced


# ----------------------------------------------------------------------------- 1. defaults unchanged
@pytest.mark.gpu
def test_defaults_equal_vsr_sample():
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"])
    V, T, b = fx["dims_obj"].vocab_size, fx["dims_obj"].seq_len, fx["det"].size(0)
    ref = m.sample_rl(*dev, seed=77)
    eng = m._engine()
    out = [torch.empty((b, T), device=DEV, dtype=dt) for dt in (torch.long, torch.long, torch.float32, torch.float32)]
    assert eng.lib.vsr_sample(eng.handle, 77, *[x.data_ptr() for x in out], None) == 0
    from vsrdec._lib import VsrSampleParams
    out_ex = [torch.empty_like(x) for x in out]
    prm = VsrSampleParams(77, 1, 1.0, 0, 1.0, 0, 0)
    assert eng.lib.vsr_sample_ex(eng.handle, ctypes.byref(prm), *[x.data_ptr() for x in out_ex], None) == 0
    torch.cuda.synchronize()
    for a, c in zip(out, out_ex):
        assert torch.equal(a, c)
    assert torch.equal(ref[0][0], out[0]) and torch.equal(ref[0][1], out[1])
    assert torch.equal(ref[1][0], out[2]) and torch.equal(ref[1][1], out[3])
    for kw in (dict(n=1), dict(top_k=V), dict(top_k=V + 5), dict(top_p=1.0), dict(temperature=1.0, top_k=0, top_p=1.0)):
        got = m.sample_rl(*dev, seed=77, **kw)
        for x, y in zip(got[0] + got[1], ref[0] + ref[1]):
            assert torch.equal(x, y), kw


# ----------------------------------------------------------------------------- 2. draw independence
def _expand(statics, reps, b):
    return tuple(s.repeat((reps,) + (1,) * (s.dim() - 1))[:b] if s is not None else None for s in statics)


@pytest.mark.gpu
@pytest.mark.parametrize("rows", ["small_a", "1150"])
def test_draw_j_does_not_depend_on_n(rows):
    fx, m = _small_a()
    statics = (fx["det"], fx["det_seqs"])
    if rows == "1150":         # 230 captions x 5 draws: the CTA-pair GEMMs; n = 1 and 2 stay below them
        statics = _expand(statics, 40, 230)
    dev = _cuda(*statics)
    for kw in (dict(), dict(temperature=0.7, top_p=0.9), dict(top_k=5, temperature=2.0)):
        full = m.sample_rl(*dev, seed=5, n=5, **kw)
        for nn in (1, 2, 3, 4):
            part = m.sample_rl(*dev, seed=5, n=nn, **kw)
            for x, y in zip(full[0] + full[1], part[0] + part[1]):
                y = y.unsqueeze(1) if nn == 1 else y
                assert torch.equal(x[:, :nn], y), (rows, kw, nn)
        w = full[0][0]
        assert len({tuple(r) for r in w[:, :, 0].tolist()}) > 1        # the draws differ


# ----------------------------------------------------------------------------- 3. support along the trajectory
@pytest.mark.gpu
@pytest.mark.parametrize("tau,top_k,top_p", [
    (1.0, 1, 1.0), (1.0, 5, 1.0), (1.0, 40, 1.0), (1.0, 0, 0.3), (1.0, 0, 0.9), (0.5, 0, 1.0), (2.0, 0, 1.0),
    (0.5, 5, 0.9), (2.0, 40, 0.3), (2.0, 40, 0.9), (1.0, 5, 0.3), (0.5, 1, 0.9)])
def test_draws_lie_in_the_truncated_set(tau, top_k, top_p):
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    statics = (fx["det"], fx["det_seqs"])
    n = 4
    res = m.sample_rl(*_cuda(*statics), seed=11, n=n, temperature=tau, top_k=top_k, top_p=top_p)
    torch.cuda.synchronize()
    assert res[0][0].shape == (statics[0].size(0), n, d.seq_len)
    _check_support(W, d, statics, res, n, tau, top_k, top_p)


# ----------------------------------------------------------------------------- 4. distribution
def _safe_top_p(lp0, tau, top_k, target):
    """A top_p near `target` with no caption's cumulative-mass point within 1e-3 of it."""
    for delta in [0.0] + [s * 0.0005 * i for i in range(1, 200) for s in (1, -1)]:
        p = target + delta
        N, V = lp0.shape
        k = V if top_k == 0 else min(top_k, V)
        slp = torch.sort(lp0.double(), 1, descending=True).values[:, :k] / tau
        q = torch.softmax(slp, 1)
        if float((q.cumsum(1) - p).abs().min()) > 1e-3:
            return p
    raise AssertionError("no safe top_p")


@pytest.mark.gpu
@pytest.mark.parametrize("tau,top_k,top_p", [(0.5, 0, 1.0), (1.0, 5, 1.0), (1.0, 0, 0.9), (2.0, 40, 0.9)])
def test_first_step_distribution(tau, top_k, top_p):
    """n = 3000 draws per caption in one call; chi-square of the first-step words against the reference distribution
    (rare words pooled, 6-sd bound as in the parity suite)."""
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    det, ds = fx["det"], fx["det_seqs"]
    b, V, N = det.size(0), d.vocab_size, 3000
    with torch.no_grad():
        (out0, _), _ = O.decoder_step(W, d, 0, O.init_state(d, b), None, (det, ds), None, "feedback")
    if top_p < 1.0:
        top_p = _safe_top_p(out0, tau, top_k, top_p)
    probs, allowed, _ = _sets(out0, tau, top_k, top_p)
    (w, _), _ = m.sample_rl(*_cuda(det, ds), seed=3, n=N, temperature=tau, top_k=top_k, top_p=top_p)
    w0 = w[:, :, 0].cpu()
    counts = torch.zeros((b, V), dtype=torch.float64).scatter_add_(1, w0, torch.ones_like(w0, dtype=torch.float64))
    assert bool((counts[~allowed] == 0).all()), "a word outside P was drawn"
    for i in range(b):
        exp = probs[i] * N
        big = exp >= 5.0
        obs = torch.cat([counts[i][big], counts[i][~big].sum().reshape(1)])
        ex = torch.cat([exp[big], exp[~big].sum().reshape(1)])
        keep = ex > 0
        chi2 = float((((obs - ex) ** 2)[keep] / ex[keep]).sum())
        dof = max(int(keep.sum()) - 1, 1)
        assert chi2 < dof + 6.0 * (2.0 * dof) ** 0.5 + 10.0, f"caption {i}: chi2 {chi2:.1f} for {dof} dof"


# ----------------------------------------------------------------------------- 5. coupling
@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p", [(5, 1.0), (0, 0.9), (40, 0.5)])
def test_truncation_keeps_draws_that_were_inside(top_k, top_p):
    """Restricted Gumbel-max: at t = 0 and tau = 1 the truncated draw of (c, j) sees the same noise as the untruncated
    one, so wherever the untruncated word is certainly inside P the truncated draw equals it."""
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    det, ds = fx["det"], fx["det_seqs"]
    b, n = det.size(0), 300
    with torch.no_grad():
        (out0, _), _ = O.decoder_step(W, d, 0, O.init_state(d, b), None, (det, ds), None, "feedback")
    _, _, certain = _sets(out0, 1.0, top_k, top_p)
    (wu, _), _ = m.sample_rl(*_cuda(det, ds), seed=9, n=n)
    (wt, _), _ = m.sample_rl(*_cuda(det, ds), seed=9, n=n, top_k=top_k, top_p=top_p)
    wu, wt = wu[:, :, 0].cpu(), wt[:, :, 0].cpu()
    inside = certain.gather(1, wu)
    assert int(inside.sum()) >= 20
    assert torch.equal(wt[inside], wu[inside])


# ----------------------------------------------------------------------------- 6. limits of the knobs
@pytest.mark.gpu
def test_top_k_1_and_tiny_top_p_are_greedy_at_the_first_step():
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    det, ds = fx["det"], fx["det_seqs"]
    dev = _cuda(det, ds)
    gw, _ = m.test(*dev)
    with torch.no_grad():
        (out0, _), _ = O.decoder_step(W, d, 0, O.init_state(d, det.size(0)), None, (det, ds), None, "feedback")
    top2 = torch.topk(out0.double(), 2, 1).values
    untied = (top2[:, 0] - top2[:, 1]) > _tol(top2[:, 0])
    for kw in (dict(top_k=1), dict(top_p=1e-6), dict(top_k=1, temperature=0.3), dict(top_p=1e-6, temperature=3.0)):
        (w, _), _ = m.sample_rl(*dev, seed=1, n=6, **kw)
        first = w[:, :, 0]
        if "top_k" in kw:
            assert torch.equal(first, gw[:, :1].expand_as(first)), kw
        else:
            assert torch.equal(first[untied.to(DEV)], gw[:, :1].expand_as(first)[untied.to(DEV)]), kw
    # and along the device trajectories every word is the oracle's best of its row
    res = m.sample_rl(*dev, seed=2, n=3, top_k=1)
    _check_support(W, d, (det, ds), res, 3, 1.0, 1, 1.0)


# ----------------------------------------------------------------------------- 7. verb forcing
@pytest.mark.gpu
@pytest.mark.parametrize("gt", [True, False])
def test_sample_v_forces_verbs(gt):
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    verbs = fx["verbs_gt"] if gt else fx["verbs_tab"]
    statics = (fx["det"], fx["det_seqs"], verbs)
    for tau, top_k, top_p in ((1.0, 0, 1.0), (0.7, 0, 0.9), (1.0, 5, 1.0)):
        n = 3
        res = m.sample_v(_cuda(*statics), n=n, temperature=tau, top_k=top_k, top_p=top_p, gt=gt, seed=4)
        torch.cuda.synchronize()
        n_forced = _check_support(W, d, statics, res, n, tau, top_k, top_p, True, gt, fx["verb_table"])
        assert n_forced > 0


# ----------------------------------------------------------------------------- 8. driver-wide
@pytest.mark.gpu
def test_attention_half_features_and_index_form():
    fx, m = _small_a()
    det, ds = fx["det"], fx["det_seqs"]
    b, T, R = det.size(0), fx["dims_obj"].seq_len, ds.size(2)
    dev = _cuda(det, ds)
    kw = dict(seed=21, temperature=0.8, top_p=0.9)
    res5 = m.sample_rl(*dev, n=5, return_attention=True, **kw)
    res1 = m.sample_rl(*dev, n=1, return_attention=True, **kw)
    att5, att1 = res5[2], res1[2]
    assert att5["alpha"].shape == (b, 5, T, R + 1) and att5["slot"].shape == (b, 5, T)
    assert att1["alpha"].shape == (b, T, R + 1)
    assert torch.equal(att5["alpha"][:, 0], att1["alpha"]) and torch.equal(att5["slot"][:, 0], att1["slot"])
    plain = m.sample_rl(*dev, n=5, **kw)
    for x, y in zip(plain[0] + plain[1], res5[0] + res5[1]):
        assert torch.equal(x, y)
    # half-precision features equal their fp32 upcast
    for dt in (torch.float16, torch.bfloat16):
        h = (det.to(DEV, dt), ds.to(DEV, dt))
        up = (h[0].float(), h[1].float())
        a = m.sample_rl(*h, n=3, top_k=7, **kw)
        c = m.sample_rl(*up, n=3, top_k=7, **kw)
        for x, y in zip(a[0] + a[1], c[0] + c[1]):
            assert torch.equal(x, y), dt
        vb = fx["verbs_gt"].to(DEV)
        a = m.sample_v(h + (vb,), n=3, gt=True, **kw)
        c = m.sample_v(up + (vb,), n=3, gt=True, **kw)
        for x, y in zip(a[0] + a[1], c[0] + c[1]):
            assert torch.equal(x, y), dt


@pytest.mark.gpu
def test_engine_index_form_equals_materialised():
    from gpu_common import make_model
    d = O.Dims(seq_len=8, vocab_size=97, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    m = make_model(d, O.init_weights(d, seed=5))
    det, idx, verbs = O.synth_inputs_indexed(7, 9, 5, 6, 64, seed=31, n_det_range=(3, 9), real_slots=(2, 5))
    idx = torch.where(idx == -2, torch.zeros_like(idx), idx)          # detection rows and padding only
    ds = O.materialize_slots(det, idx)
    eng = m._engine()
    out = []
    for form in ("indexed", "materialised"):
        if form == "indexed":
            eng.prologue_indexed(det.to(DEV), idx.to(DEV), verbs.to(DEV))
        else:
            eng.prologue(det.to(DEV), ds.to(DEV), verbs.to(DEV))
        out.append(eng.sample(17, n=4, temperature=1.3, top_k=20, top_p=0.8, use_verbs=True, gt=True))
    for x, y in zip(out[0][0] + out[0][1], out[1][0] + out[1][1]):
        assert x.shape == (7, 4, 8) and torch.equal(x, y)


# ----------------------------------------------------------------------------- 9. vocabulary edge cases
@pytest.mark.gpu
@pytest.mark.parametrize("V", [97, 49152])
def test_vocabulary_edges(V):
    from gpu_common import make_model
    d = O.Dims(seq_len=5, vocab_size=V, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    W = O.init_weights(d, seed=8)
    W["out_fc.weight"] = W["out_fc.weight"] * 20.0          # a peaked distribution, so top-p sets stay small
    m = make_model(d, W)
    det, ds, _ = O.synth_inputs(3, 9, 5, 6, 64, seed=41, vocab_size=V, n_det_range=(3, 9), real_slots=(2, 5))
    for top_k in (0, 7, V - 1):
        for top_p in (0.5, 1.0):
            res = m.sample_rl(*_cuda(det, ds), seed=top_k + 1, n=2, top_k=top_k, top_p=top_p)
            torch.cuda.synchronize()
            _check_support(W, d, (det, ds), res, 2, 1.0, top_k, top_p)


@pytest.mark.gpu
@pytest.mark.parametrize("top_k,top_p", [(0, 0.33), (10, 1.0), (10, 0.33), (10, 0.71), (50, 0.71), (96, 0.5)])
def test_exact_ties_resolve_in_index_order(top_k, top_p):
    """Every row of out_fc is the same vector and the bias is 0, so all V logits tie exactly at every step.  The order
    (x desc, index asc) is then the index order: K = {0 .. k-1}, and with equal masses P = the first ceil(top_p * k)
    entries of K (top_p as the float32 the library receives).  The draws must fill exactly P: both boundaries fall
    inside one group of tied values and are resolved in index order."""
    from gpu_common import make_model
    d = O.Dims(seq_len=4, vocab_size=97, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    W = O.init_weights(d, seed=8)
    W["out_fc.weight"] = W["out_fc.weight"][:1].expand_as(W["out_fc.weight"]).clone()
    W["out_fc.bias"] = torch.zeros_like(W["out_fc.bias"])
    m = make_model(d, W)
    det, ds, _ = O.synth_inputs(3, 9, 5, 6, 64, seed=41, vocab_size=97, n_det_range=(3, 9), real_slots=(2, 5))
    k = 97 if top_k == 0 else top_k
    size = math.ceil(ctypes.c_float(top_p).value * k) if top_p < 1.0 else k
    (w, _), (lw, _) = m.sample_rl(*_cuda(det, ds), seed=12, n=700, top_k=top_k, top_p=top_p)
    w = w.cpu()
    assert int(w.max()) < size, (size, int(w.max()))
    assert set(w[:, :, 0].flatten().tolist()) == set(range(size))
    assert rel_close(lw.cpu(), torch.full(lw.shape, -math.log(97.0)), REL, ABS)     # the model's uniform log-prob


@pytest.mark.gpu
def test_tiny_temperature_stays_finite():
    """At temperature 1e-40 (nonzero in float32) x / temperature overflows float32; z is clamped, so the draws stay in
    the truncated set and the returned log-probs stay the model's."""
    fx, m = _small_a()
    d, W = fx["dims_obj"], fx["weights"]
    det, ds = fx["det"], fx["det_seqs"]
    for top_k, top_p in ((5, 0.9), (5, 1.0), (0, 1.0)):
        res = m.sample_rl(*_cuda(det, ds), seed=6, n=3, temperature=1e-40, top_k=top_k, top_p=top_p)
        torch.cuda.synchronize()
        (w, g), (lw, lg) = res
        assert bool(torch.isfinite(lw).all()) and bool(torch.isfinite(lg).all())
        assert int(w.min()) >= 0 and int(w.max()) < d.vocab_size
        _check_support(W, d, (det, ds), res, 3, 1.0, top_k, 1.0)       # inside K: the top-k set does not depend on tau


# ----------------------------------------------------------------------------- 10. errors
@pytest.mark.gpu
def test_invalid_arguments():
    from vsrdec import VsrError
    from vsrdec._lib import VsrSampleParams
    fx, m = _small_a()
    dev = _cuda(fx["det"], fx["det_seqs"])
    m.sample_rl(*dev, seed=1)
    eng = m._engine()
    torch.cuda.synchronize()
    bad = [dict(n=0), dict(n=-2), dict(n=1.5), dict(temperature=0.0), dict(temperature=-1.0),
           dict(temperature=float("nan")), dict(temperature=float("inf")), dict(top_k=-1), dict(top_k=2.0),
           dict(top_p=0.0), dict(top_p=-0.1), dict(top_p=1.5), dict(top_p=float("nan")), dict(temperature=1e-50),
           dict(top_p=1e-50), dict(temperature=1e39)]
    launches = eng.launch_count()
    for kw in bad:
        with pytest.raises(VsrError):
            m.sample_rl(*dev, seed=1, **kw)
        with pytest.raises(VsrError):
            m.sample_v(dev + (fx["verbs_gt"].to(DEV),), seed=1, **kw)
        with pytest.raises(VsrError):
            eng.sample(1, **kw)
    with pytest.raises(VsrError):
        m.sample_v(dev, seed=1)                              # no verbs
    with pytest.raises(VsrError):
        eng.sample(1, use_verbs=True)                        # the prologue has no verbs tensor
    assert eng.launch_count() == launches                    # nothing was launched
    b, T = dev[0].size(0), fx["dims_obj"].seq_len
    out = [torch.empty((b, 2, T), device=DEV, dtype=dt) for dt in (torch.long, torch.long, torch.float32, torch.float32)]
    ptrs = [x.data_ptr() for x in out]
    lib = eng.lib
    for args in ((1, 0, 1.0, 0, 1.0, 0, 0), (1, 2, 0.0, 0, 1.0, 0, 0), (1, 2, float("inf"), 0, 1.0, 0, 0),
                 (1, 2, float("nan"), 0, 1.0, 0, 0), (1, 2, 1.0, -1, 1.0, 0, 0), (1, 2, 1.0, 0, 0.0, 0, 0),
                 (1, 2, 1.0, 0, 1.5, 0, 0), (1, 2, 1.0, 0, 1.0, 1, 0)):
        prm = VsrSampleParams(*args)
        assert lib.vsr_sample_ex(eng.handle, ctypes.byref(prm), *ptrs, None) == -1, args     # VSR_EINVAL
    prm = VsrSampleParams(1, 2, 1.0, 0, 1.0, 0, 0)
    assert lib.vsr_sample_ex(eng.handle, None, *ptrs, None) == -1
    assert lib.vsr_sample_ex(eng.handle, ctypes.byref(prm), ptrs[0], None, ptrs[2], ptrs[3], None) == -1
    assert lib.vsr_sample_ex(eng.handle, ctypes.byref(prm), *ptrs, None) == 0
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- 11. CPU-only
def _header():
    return open(os.path.join(ROOT, "include", "vsrdec.h")).read()


def test_header_declares_vsr_sample_ex_and_the_struct_matches_ctypes():
    src = re.sub(r"/\*.*?\*/", "", _header(), flags=re.S)
    assert "vsr_sample_ex" in set(re.findall(r"\b(vsr_[a-z_0-9]+)\s*\(", src))
    body = re.search(r"typedef struct VsrSampleParams \{(.*?)\} VsrSampleParams;", src, flags=re.S).group(1)
    fields = re.findall(r"(uint64_t|int32_t|float)\s+(\w+);", body)
    size_of = {"uint64_t": 8, "int32_t": 4, "float": 4}
    off, offsets = 0, []
    for ty, name in fields:                               # natural alignment, as the C compiler lays it out
        off = (off + size_of[ty] - 1) // size_of[ty] * size_of[ty]
        offsets.append((name, off))
        off += size_of[ty]
    size = (off + 7) // 8 * 8
    from vsrdec._lib import VsrSampleParams
    assert [(n, getattr(VsrSampleParams, n).offset) for n, _ in VsrSampleParams._fields_] == offsets
    assert ctypes.sizeof(VsrSampleParams) == size == 32
    import vsrdec
    assert "vsr_sample_ex" in vsrdec.EXPORTED_SYMBOLS


def test_library_exports_vsr_sample_ex():
    import vsrdec
    path = vsrdec.library_path()
    if not os.path.isfile(path):
        pytest.skip("libvsrdec.so is not built")
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    assert "vsr_sample_ex" in set(re.findall(r" T (vsr_[a-z_0-9]+)", out))


def test_sampling_signatures():
    import inspect
    from models import ControllableCaptioningModel
    from models.CaptioningModel import CaptioningModel
    defaults = dict(n=1, temperature=1.0, top_k=0, top_p=1.0)
    for fn in (CaptioningModel.sample_rl, ControllableCaptioningModel.sample_rl):
        ps = inspect.signature(fn).parameters
        for k, v in dict(defaults, seed=None, return_attention=False).items():
            assert ps[k].default == v, (fn, k)
    ps = list(inspect.signature(ControllableCaptioningModel.sample_rl).parameters)
    assert ps[:5] == ["self", "detections", "ctrl_det_seqs_test", "seed", "return_attention"]
    sv = inspect.signature(CaptioningModel.sample_v).parameters
    assert list(sv)[:2] == ["self", "statics"]
    for k, v in dict(defaults, gt=False, seed=None, return_attention=False).items():
        assert sv[k].default == v and sv[k].kind == inspect.Parameter.KEYWORD_ONLY, k
    assert hasattr(ControllableCaptioningModel, "sample_v")
    from vsrdec import DecoderEngine
    es = inspect.signature(DecoderEngine.sample).parameters
    for k, v in dict(defaults, use_verbs=False, gt=False).items():
        assert es[k].default == v, k


def test_argument_check_without_a_device():
    from vsrdec import VsrError
    from vsrdec.engine import check_sample_args
    check_sample_args(1, 1.0, 0, 1.0)
    check_sample_args(3000, 0.01, 49152, 1e-6)
    for args in ((0, 1.0, 0, 1.0), (True, 1.0, 0, 1.0), (1, math.inf, 0, 1.0), (1, 1.0, -3, 1.0), (1, 1.0, 0, 0.0),
                 (1, 1.0, 0, 1.0001), (1, "x", 0, 1.0), (1, 1e-50, 0, 1.0), (1, 1e39, 0, 1.0), (1, 1.0, 0, 1e-50)):
        with pytest.raises(VsrError):
            check_sample_args(*args)
    check_sample_args(1, 1e-40, 0, 1.0)                       # nonzero in float32
    check_sample_args(4, 1.0, 0, 1.0, b=2 ** 28)
    with pytest.raises(VsrError):
        check_sample_args(5, 1.0, 0, 1.0, b=2 ** 28)         # more than 2^30 rows
