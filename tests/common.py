"""Shared helpers for the test-suite (fixture loading, tie-aware comparisons)."""
import os

import torch

from oracle import vsr_oracle as O
from oracle.ssp_oracle import checksum  # noqa: F401  (the golden fixtures' checksum)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_golden(name):
    fx = torch.load(os.path.join(GOLDEN, name), weights_only=False)
    fx["dims_obj"] = O.Dims(**fx["dims"])
    if "det_seqs" in fx and "ctrl_rule" in fx:
        ds = fx["det_seqs"]
        b, L = ds.shape[0], ds.shape[1]
        T = fx["dims"]["seq_len"]
        ctrl = torch.zeros((b, T) + tuple(ds.shape[2:]))
        for t in range(T):
            ctrl[:, t] = ds[:, min(t // 2, L - 1)]
        fx["ctrl"] = ctrl
    return fx


def rel_close(a, b, rel=1e-3, abs_floor=1e-4):
    """|a-b| <= rel*|b| + abs_floor element-wise (north-star tolerance for log-probs)."""
    a, b = a.double(), b.double()
    return bool(((a - b).abs() <= rel * b.abs() + abs_floor).all())


def max_rel_err(a, b, abs_floor=1e-4):
    a, b = a.double(), b.double()
    return float(((a - b).abs() / (b.abs() + abs_floor)).max())


def tol_ratio(a, b, rel=1e-3, abs_floor=1e-4):
    """max |a-b| / (rel*|b| + abs_floor): <= 1 means inside the north-star tolerance.  The additive
    floor matters for log-probs near 0 (e.g. log(1 - e^-14) ~ -5e-7), where fp32 evaluation of
    log(1 + eps) is itself quantised to ~1e-7 and a purely relative criterion is meaningless."""
    a, b = a.double(), b.double()
    return float(((a - b).abs() / (rel * b.abs() + abs_floor)).max())


# ----------------------------------------------------------------------------- tie-aware beam check
class BeamVerdict:
    def __init__(self):
        self.decisions = 0          # (step, caption) pairs checked
        self.in_band = 0            # pairs whose k-th / (k+1)-th oracle candidates are closer than the band
        self.set_mismatch = 0       # pairs where the device's selected set differs from the oracle's top-k set
        self.violations = []        # hard failures (outside the tie band)
        self.max_score_err = 0.0
        self.max_out_rel = 0.0      # per-step log-prob error as a fraction of the tolerance
        self.max_gate_rel = 0.0     #   |dev - oracle| / (1e-3*|oracle| + 1e-4); <= 1 passes
        self.max_out_abs = 0.0
        self.max_gate_abs = 0.0
        self.band_caption = None    # bool (b,): the caption had at least one decision (or its final ordering) inside the band

    def decisive_captions(self):
        """Captions whose every top-k decision AND final beam ordering were outside the tie band: on these the device's
        tokens must equal the free-running reference's, bit for bit."""
        return ~self.band_caption

    def summary(self):
        return (f"decisions={self.decisions} in_tie_band={self.in_band} set_mismatch={self.set_mismatch} "
                f"violations={len(self.violations)} max_score_err={self.max_score_err:.3e} "
                f"out_err(tol-frac/abs)={self.max_out_rel:.3e}/{self.max_out_abs:.3e} "
                f"gate_err(tol-frac/abs)={self.max_gate_rel:.3e}/{self.max_gate_abs:.3e}")


def verify_device_beam(W, d, statics, eos, k, hist, use_verbs=False, gt=False, verb_table=None,
                       step_out=None, step_gate=None, band_abs=2e-3, band_rel=1e-4):
    """Replay the DEVICE's beam trajectory (hist = parent, word, gate, score each (T,b,k), CPU)
    through the oracle and check, at every step and caption, that the device's selection is a
    valid top-k of the ORACLE's candidate scores up to a tie band:
      * every selected candidate scores >= (oracle k-th best) - band,
      * every candidate scoring > (oracle k-th best) + band was selected,
      * the device's accumulated scores equal the oracle's at the selected candidates (<= band_abs + 2*band_rel*|score|).
    Optionally also compares the per-step log-probs (step_out (T,b*k,V), step_gate (T,b*k,2)).
    band = band_abs + band_rel*|score|: a tenth of the north star's 1e-3 relative tolerance on the log-probs the scores
    are sums of (fp32 accumulated scores reach ~ -200, where one ulp is 1.5e-5; with out_fc sharpened x100 the
    f16+f8x2 GEMM mode's per-step log-prob error is up to ~1e-3 absolute and drifts to a few 1e-3 over 20 steps).
    """
    parent, word, gate, score = [x.cpu() for x in hist]
    T, b, _ = parent.shape
    V = d.vocab_size
    forced = O.BeamTrace([parent[t].long() for t in range(T)], [word[t].long() for t in range(T)],
                         [gate[t].long() for t in range(T)], [], [], [], [])
    v = BeamVerdict()

    def hook(t, out, gate_lp, flat):
        cur = flat.size(1) // (2 * V)
        sel = parent[t].long() * (2 * V) + word[t].long() * 2 + gate[t].long()      # (b,k)
        sel_sc = torch.gather(flat, 1, sel)
        top = torch.topk(flat, k + 1, dim=1).values
        kth, nxt = top[:, k - 1], top[:, k]
        band = band_abs + band_rel * kth.abs()
        v.decisions += b
        inb = (kth - nxt) <= band
        # the ORDER of the selected candidates matters too (slot order decides the final sort's tie-breaks and which
        # beam is "best"): adjacent selected scores closer than the band make the caption non-decisive
        if k > 1:
            inb = inb | ((top[:, :k - 1] - top[:, 1:k]) <= band.unsqueeze(1)).any(1)
        v.in_band += int(((kth - nxt) <= band).sum())
        v.band_caption = inb.clone() if v.band_caption is None else (v.band_caption | inb)
        oracle_sel = torch.topk(flat, k, dim=1).indices
        v.set_mismatch += int((oracle_sel.sort(1).values != sel.sort(1).values).any(1).sum())
        low = sel_sc < (kth - band).unsqueeze(1)
        for c in torch.nonzero(low.any(1)).flatten().tolist():
            v.violations.append(f"t={t} caption={c}: selected score {sel_sc[c].tolist()} below k-th {float(kth[c])}")
        must = flat > (kth + band).unsqueeze(1)                                   # decisive candidates
        picked = torch.zeros_like(must)
        picked.scatter_(1, sel, True)
        miss = (must & ~picked).any(1)
        for c in torch.nonzero(miss).flatten().tolist():
            v.violations.append(f"t={t} caption={c}: a decisive candidate was not selected")
        err = (score[t] - sel_sc).abs()
        v.max_score_err = max(v.max_score_err, float(err.max()))
        bad = err > (band_abs + 2 * band_rel * sel_sc.abs())
        for c in torch.nonzero(bad.any(1)).flatten().tolist():
            v.violations.append(f"t={t} caption={c}: device score {score[t, c].tolist()} vs oracle {sel_sc[c].tolist()}")
        if step_out is not None:
            n = out.size(0)
            dv = step_out[t, :n].cpu()
            v.max_out_abs = max(v.max_out_abs, float((dv - out).abs().max()))
            v.max_out_rel = max(v.max_out_rel, tol_ratio(dv, out))
        if step_gate is not None:
            n = gate_lp.size(0)
            dg = step_gate[t, :n].cpu()
            v.max_gate_abs = max(v.max_gate_abs, float((dg - gate_lp).abs().max()))
            v.max_gate_rel = max(v.max_gate_rel, tol_ratio(dg, gate_lp))

    with torch.no_grad():
        outs, lps = O.beam_search(W, d, statics, eos, k, k, use_verbs=use_verbs, gt=gt, verb_table=verb_table,
                                  forced=forced, step_hook=hook)
    return v, outs, lps


def check_returned_beams(tag, d, hist, out_size, dev, o_outs, o_lps, rel=1e-3, abs_floor=1e-4, band_abs=2e-3, band_rel=1e-4):
    """The captions a beam search returns are the unrolls of its final beams in the order of their final scores.  The
    oracle, replaying the device's trajectory, orders the final beams by ITS scores: rank r of the device must be the
    oracle's rank r, or a beam whose final score ties with it inside the band (final scores of different beams routinely
    agree to ~1e-5 at |score| ~ 170 with raw random-init weights, and to ~1e-3 with the x100-sharpened head).
    dev = (words, gates, lp_words, lp_gates) as returned (b, out_size, T) or (b, T); o_* = the oracle's (b, k, T)."""
    w, g, lw, lg = [x.cpu() for x in dev]
    T = d.seq_len
    b = w.shape[0]
    w, g, lw, lg = [x.reshape(b, out_size, T) for x in (w, g, lw, lg)]
    ow, og = o_outs[0].reshape(b, -1, T), o_outs[1].reshape(b, -1, T)
    olw, olg = o_lps[0].reshape(b, -1, T), o_lps[1].reshape(b, -1, T)
    dev_final = hist[3][-1].cpu().sort(1, descending=True).values          # device scores of the final beams, best first
    swapped = 0
    for c in range(b):
        for r in range(out_size):
            hit = [q for q in range(ow.size(1)) if torch.equal(ow[c, q], w[c, r]) and torch.equal(og[c, q], g[c, r])]
            assert hit, f"{tag}: caption {c} rank {r} is not the unroll of any final beam of its own trajectory"
            q = min(hit, key=lambda x: abs(x - r))
            band = band_abs + band_rel * float(dev_final[c, r].abs())
            assert q == r or abs(float(dev_final[c, r] - dev_final[c, q])) <= band, f"{tag}: caption {c} returned beam {q} at rank {r}"
            swapped += int(q != r)
            assert rel_close(lw[c, r], olw[c, q], rel, abs_floor) and rel_close(lg[c, r], olg[c, q], rel, abs_floor), \
                f"{tag}: caption {c} rank {r}: returned log-probs differ from the oracle's"
    return swapped


from tools.synth import synth_eval_captions  # noqa: E402,F401  (shared with bench.py)
