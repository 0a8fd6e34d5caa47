"""The decoder step and the decode drivers against a float64 run of the oracle, at trained-like parameters and feature
magnitudes, in every GEMM mode (the default f16+f8x2, VSRDEC_GEMM=f16x3 and the fp32 FFMA twin VSRDEC_GEMM=simt).

The constructor's initialisation hides whole classes of mistakes: all ten bias tensors are zero, so a dropped bias term,
two gates swapped in a packed bias or a bias that leaks into a pad column give the same numbers as the correct packing.
`trained_like` rewrites the parameters (every bias N(0, 0.1), LSTM forget-gate biases +1, every weight matrix scaled by
its own factor from {0.5, 1, 2}, out_fc.bias shifted to about -30 so that a pad column's logit 0 would win any top-k or
log-sum-exp it leaked into) and loads them through load_state_dict, the path a checkpoint takes.

The reference is oracle/vsr_oracle.py, unchanged, fed float64 parameters and inputs.  Each bound below is a fraction of
the output scale of the GEMM that produces the quantity, per row; the float32 oracle must meet the same bound on the same
inputs.  The last test (no GPU needed) ties the float64 oracle at trained-like parameters to the float32 oracle and the
golden vectors of the unmodified reference."""
import pytest
import torch
import torch.nn.functional as F

from common import check_returned_beams, load_golden, rel_close, verify_device_beam
from oracle import vsr_oracle as O

DEV = "cuda:0"
MODES = ["f16+f8x2", "f16x3", "simt"]
MODE_IDS = ["default", "f16x3", "simt"]
KIND = {"f16+f8x2": "tcgen05-f16+f8x2", "f16x3": "tcgen05-f16x3", "simt": "simt-fp32"}

# Error of one GEMM output, as a fraction of the GEMM's output scale (max |output| of the row):
#   simt:     fp32 FFMA over K <= 4096 terms, as the float32 oracle itself: sqrt(K) * 2^-24 = 2^-18;
#   f16x3:    hi + lo carries 22 bits (2^-22), plus the tensor-core accumulation TC_ACC below;
#   f16+f8x2: the residual products hi8 * W_lo8 and lo8 * W_hi8 carry e4m3 operands (3 mantissa bits) on residuals of
#             2^-11 relative, so each product is off by up to 2^-4 * 2^-11 = 2^-15 of itself; plus TC_ACC.
# TC_ACC: the tensor cores do not accumulate like an fp32 FFMA chain.  Each k-block's products are aligned to the
# accumulator and truncated, up to 2^-24 of the running sum per 16-element k-block and with one sign, so K / 16 * 2^-24
# = 2^-16 for K <= 4096.  Measured on a B200 (1000 W) with the fp32-level 2^-18 in its place, f16x3 reached 2.6x that
# bound (c1, c2, out and gate), while simt stayed at 0.27x and f16+f8x2 showed the same absolute errors as f16x3:
# the error comes from the accumulator the two tensor-core modes share, not from their operand formats.
TC_ACC = 2.0 ** -16
EPS = {"f16+f8x2": 2.0 ** -15 + TC_ACC, "f16x3": 2.0 ** -22 + TC_ACC, "simt": 2.0 ** -18}
# Propagation from the GEMM output δ to the compared quantity (sigmoid' <= 1/4, tanh' <= 1, |f|, |i|, |o| <= 1):
#   c' = f c + i g:   δc' <= (1/4 |c| + 1/4 + 1) δ;   h' = o tanh(c'):   δh' <= δ/4 + δc'
#   cell 2 also carries the error of its inputs h1' and att, of the same order as its own: x2
#   log-softmax: z_i - lse(z) moves by up to 2 max δz; the logits carry h2''s error as well: x2
def c_factor(c_old):
    return 1.25 + c_old.abs().amax(1) / 4


def h_factor(c_old):
    return 1.5 + c_old.abs().amax(1) / 4


CELL2_INPUTS = 2.0
LOGSOFTMAX = 4.0
# gate log-probs: log-softmax of two logits that are sums over the attention size of att_g * tanh(GEMM-C + ha) and
# att_a * tanh(P + ha): the output scale is that of the logits themselves (max(1, |log-prob|) of the row), x4 as above
GATE = 4.0
# Whole decodes: the contract's 1e-3 relative + 1e-4 absolute on log-probs, with verify_device_beam's tie band on top-k.
REL, ABS = 1e-3, 1e-4


# ----------------------------------------------------------------------------- parameters
def trained_like(d, seed, s_fc=1.0, out_shift=-30.0):
    """O.init_weights(d, seed) rewritten with trained-like values (see the module docstring); s_fc.weight and s_fc.bias
    are multiplied by `s_fc`, which moves the sentinel s_fc(s_t) to a chosen magnitude.  float32 tensors."""
    W = O.init_weights(d, seed)
    g = torch.Generator().manual_seed(seed + 7)
    H = d.rnn_size
    out = {}
    for k, v in W.items():
        if v.dim() == 1:
            t = torch.randn(v.shape, generator=g, dtype=torch.float64) * 0.1
            if k in ("lstm_cell_1.bias_ih", "lstm_cell_2.bias_ih"):
                t[H:2 * H] += 1.0                      # forget gate (gate order i, f, g, o)
            if k == "out_fc.bias":
                t += out_shift
        else:
            t = v.double() * (0.5, 1.0, 2.0)[int(torch.randint(0, 3, (1,), generator=g))]
        if k.startswith("s_fc."):
            t = t * s_fc
        out[k] = t.float().contiguous()
    return out


def _f64(x):
    if isinstance(x, dict):
        return {k: v.double() for k, v in x.items()}
    return tuple(t.double() if t.is_floating_point() else t for t in x)


_MODELS = {}


def _model(monkeypatch, mode, d, W, table=None):
    """The drop-in model of dims `d` in GEMM mode `mode`, holding parameters W.  One model per (mode, dims) is kept; a
    later W reaches it through load_state_dict, i.e. through the native weight reload."""
    from gpu_common import make_model
    key = (mode, d)
    m = _MODELS.get(key)
    if m is None:
        if mode == "f16+f8x2":
            monkeypatch.delenv("VSRDEC_GEMM", raising=False)
        else:
            monkeypatch.setenv("VSRDEC_GEMM", mode)            # read when the native handle is created
        m = make_model(d, W, table)
        m._engine()
        _MODELS[key] = m
    else:
        m.load_state_dict(W)
        m.verb_2_vob_all = table or {}
    assert m._eng.gemm_kind() == KIND[mode]
    return m


def _cuda(xs):
    return tuple(x.to(DEV) for x in xs)


# ----------------------------------------------------------------------------- inputs
def step_inputs(d, b, R, seed, L=6, D=30, sentinel_only=False, verbs=False):
    """Statics (det, det_seqs, verbs), an explicit state and the previous outputs of step 1.
    Ragged slots (1..R valid rows), every third row's slot 0 empty (the sentinel is its only region), h in [-1, 1],
    c in [-20, 20] (tanh(c) saturated on most units)."""
    det, ds, vb = O.synth_inputs(b, D, L, R, d.det_feat_size, seed=seed, vocab_size=d.vocab_size,
                                 n_det_range=(min(5, D), D), real_slots=(2, L), verb_slots=(1,) if verbs else (),
                                 verb_vocab_id=17)
    if sentinel_only:
        ds.zero_()
    else:
        ds[::3, 0] = 0
    g = torch.Generator().manual_seed(seed + 1)
    H = d.rnn_size
    h1, h2 = (torch.rand((b, H), generator=g) * 2 - 1 for _ in range(2))
    c1, c2 = (torch.rand((b, H), generator=g) * 40 - 20 for _ in range(2))
    ptr = torch.randint(0, L, (b,), generator=g)
    prev = (torch.randint(0, d.vocab_size, (b,), generator=g), torch.randint(0, 2, (b,), generator=g))
    return (det, ds, vb), ((h1, c1), (h2, c2), ptr), prev


def ref_step(W, d, state, prev, statics, use_verbs, gt=True):
    """One oracle step (t = 1, feedback) plus what the bounds need: max |pre-activation| per row of each LSTM cell
    (GEMM-A, GEMM-D), max |out_fc . h2'| per row (the vocabulary GEMM) and the attended features att."""
    rec = []
    cell = O._lstm_cell

    def recording_cell(x, h, c, w_ih, w_hh, b_ih, b_hh):
        pre = F.linear(x, w_ih, b_ih) + F.linear(h, w_hh, b_hh)
        rec.append((x, pre.abs().amax(1)))
        return cell(x, h, c, w_ih, w_hh, b_ih, b_hh)

    O._lstm_cell = recording_cell
    try:
        with torch.no_grad():
            (out, gate), ((h1, c1), (h2, c2), _) = O.decoder_step(W, d, 1, state, prev, statics, None, "feedback",
                                                                    use_verbs=use_verbs, gt=gt)
    finally:
        O._lstm_cell = cell
    H, Fd = d.rnn_size, d.det_feat_size
    att = rec[1][0][:, H:H + Fd]
    s_e = F.linear(h2, W["out_fc.weight"]).abs().amax(1)
    return dict(h1=h1, c1=c1, h2=h2, c2=c2, out=out, gate=gate, s_a=rec[0][1], s_d=rec[1][1], s_e=s_e, att=att)


def step_bounds(mode, r, state):
    """Per-row bound of each compared quantity (see the constants above)."""
    (_, c1), (_, c2), _ = state
    e = EPS[mode]
    one = torch.ones_like(r["s_a"])
    return dict(h1=e * r["s_a"] * h_factor(c1), c1=e * r["s_a"] * c_factor(c1),
                h2=e * CELL2_INPUTS * r["s_d"] * h_factor(c2), c2=e * CELL2_INPUTS * r["s_d"] * c_factor(c2),
                out=e * LOGSOFTMAX * torch.maximum(r["s_e"], one),
                gate=e * GATE * torch.maximum(r["gate"].abs().amax(1), one))


def bound_ratio(got, ref, bound):
    """max over rows of max |got - ref| / bound (bound per row)."""
    err = (got.double() - ref.double()).abs().reshape(ref.shape[0], -1).amax(1)
    return float((err / bound).max())


def dev_step(m, state, prev, statics, use_verbs, gt=True):
    st = ((state[0][0].to(DEV), state[0][1].to(DEV)), (state[1][0].to(DEV), state[1][1].to(DEV)), state[2].to(DEV))
    pv = (prev[0].to(DEV), prev[1].to(DEV))
    fn = m.step_v if use_verbs else m.step
    kw = dict(gt=gt) if use_verbs else {}
    (out, gate), ((h1, c1), (h2, c2), _) = fn(1, st, pv, statics, None, mode="feedback", **kw)
    torch.cuda.synchronize()
    return dict(h1=h1.cpu(), c1=c1.cpu(), h2=h2.cpu(), c2=c2.cpu(), out=out.cpu(), gate=gate.cpu())


QUANTITIES = ("h1", "c1", "h2", "c2", "out", "gate")


def check_step(tag, mode, got, W, d, state, prev, statics, use_verbs, gt=True):
    """Device step `got` against the float64 oracle; the float32 oracle must meet the same bounds.  Returns the float64
    reference and the bound ratios of the device."""
    r64 = ref_step(_f64(W), d, (_f64(state[0]), _f64(state[1]), state[2]), prev, _f64(statics), use_verbs, gt)
    r32 = ref_step(W, d, state, prev, statics, use_verbs, gt)
    bounds = step_bounds(mode, r64, state)
    dev = {q: bound_ratio(got[q], r64[q], bounds[q]) for q in QUANTITIES}
    o32 = {q: bound_ratio(r32[q], r64[q], bounds[q]) for q in QUANTITIES}
    print(f"DECODER-F64 {tag} [{mode}] max|att| {float(r64['att'].abs().max()):.1f}: device / bound "
          + " ".join(f"{q} {dev[q]:.3f}" for q in QUANTITIES) + " | fp32 oracle / bound "
          + " ".join(f"{q} {o32[q]:.3f}" for q in QUANTITIES))
    for q in QUANTITIES:
        assert o32[q] <= 1.0, (tag, mode, "fp32 oracle", q, o32[q])
    for q in QUANTITIES:
        assert dev[q] <= 1.0, (tag, mode, "device", q, dev[q])
    return r64, dev


# ----------------------------------------------------------------------------- 1. single steps with explicit state
FULL = O.Dims()
ODD_V = O.Dims(vocab_size=97)
# (tag, dims, rows, regions per slot, sentinel only, verb slots)
STEP_CASES = [
    ("b1-sentinel-only", FULL, 1, 20, True, False),
    ("b7-ragged", FULL, 7, 20, False, False),
    ("b7-R64", FULL, 7, 64, False, False),            # R + 1 > 32: the attention's serial softmax
    ("b129-verbs", FULL, 129, 20, False, True),       # two row tiles, verb slots forced (gt)
    ("b640-pair", FULL, 640, 20, False, False),       # PAIR_MIN_ROWS: GEMM-B, D+C and E on the CTA-pair kernel
    ("b7-V97", ODD_V, 7, 20, False, True),
]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("case", STEP_CASES, ids=[c[0] for c in STEP_CASES])
def test_step_at_trained_like_parameters(monkeypatch, mode, case):
    tag, d, b, R, sent, verbs = case
    W = trained_like(d, seed=11)
    m = _model(monkeypatch, mode, d, W)
    statics, state, prev = step_inputs(d, b, R, seed=100 + b + R, sentinel_only=sent, verbs=verbs)
    got = dev_step(m, state, prev, _cuda(statics), verbs)
    check_step(tag, mode, got, W, d, state, prev, statics, verbs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_step_after_weight_reload(monkeypatch, mode):
    """Parameters that reach the packed copy through vsr_load_weights after a first decode with other values."""
    d = FULL
    m = _model(monkeypatch, mode, d, trained_like(d, seed=12))
    statics, state, prev = step_inputs(d, 7, 20, seed=41)
    dev_step(m, state, prev, _cuda(statics), False)
    W = trained_like(d, seed=13)
    m.load_state_dict(W)
    got = dev_step(m, state, prev, _cuda(statics), False)
    check_step("reload", mode, got, W, d, state, prev, statics, False)


# ----------------------------------------------------------------------------- 2. feature and sentinel magnitude
ATT_TARGETS = [4.0, 30.0, 100.0, 250.0]
HOT = 16


def _max_att(W, d, state, prev, statics):
    return float(ref_step(_f64(W), d, (_f64(state[0]), _f64(state[1]), state[2]), prev, _f64(statics), False)["att"]
                 .abs().max())


def magnitude_case(d, route, target, seed=51, b=16):
    """Parameters and inputs whose attended features att reach max |att| = target (within 10 %, at most 255), either
    through the region features (scaled, then rounded to fp16 so that the fp16 features equal them exactly) or through
    the sentinel (s_fc scaled; every slot empty, so att is the sentinel)."""
    statics, state, prev = step_inputs(d, b, 20, seed=seed, sentinel_only=(route == "s_fc"))
    det, ds, vb = statics
    if route == "s_fc":
        W1 = trained_like(d, seed=14)
        k = target / _max_att(W1, d, state, prev, statics)     # att = sentinel, linear in the s_fc parameters
        W = trained_like(d, seed=14, s_fc=k)
        feats = (det.half().float(), ds.half().float())
    else:
        # the first HOT feature columns of every real region row carry the same value a, the other columns are
        # relu(randn); att's hot columns are then a times the attention mass on the regions
        W = trained_like(d, seed=14)

        def feats_at(a):
            out = []
            for x in (det, ds):
                x = x.clone()
                hot = x[..., :HOT]
                hot[x.sum(-1) != 0] = a
                out.append(x.half().float())
            return tuple(out)

        a = target
        for _ in range(3):                                     # the attention moves as the features grow
            a = min(a * target / _max_att(W, d, state, prev, feats_at(a) + (vb,)), 255.0)
        feats = feats_at(a)
    statics = feats + (vb,)
    got = _max_att(W, d, state, prev, statics)
    assert 0.9 * target <= got <= min(1.1 * target, 255.0), (route, target, got)
    return W, statics, state, prev


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("route", ["features", "s_fc"])
@pytest.mark.parametrize("target", ATT_TARGETS)
def test_step_at_attended_feature_magnitude(monkeypatch, mode, route, target):
    """At max |att| of about 4 (synthetic relu(randn) features), 30, 100 and 250.  The fp16 copy of the features decodes
    to the same bits as the fp32 one (the fp32 values are fp16 values)."""
    d = FULL
    W, statics, state, prev = magnitude_case(d, route, target)
    m = _model(monkeypatch, mode, d, W)
    got = dev_step(m, state, prev, _cuda(statics), False)
    check_step(f"att~{target:g} via {route}", mode, got, W, d, state, prev, statics, False)
    if mode != "simt":            # the FFMA twin refuses half-precision features
        half = (statics[0].to(DEV, torch.float16), statics[1].to(DEV, torch.float16), statics[2].to(DEV))
        got_h = dev_step(m, state, prev, half, False)
        for q in QUANTITIES:
            assert torch.equal(got_h[q], got[q]), (route, target, mode, q)


@pytest.mark.gpu
@pytest.mark.parametrize("route", ["features", "s_fc"])
@pytest.mark.parametrize("target", [4.0, 250.0])
def test_tensor_core_modes_against_simt(monkeypatch, route, target):
    """The two tensor-core modes against the FFMA twin on the same step, within the sum of both modes' bounds."""
    d = FULL
    W, statics, state, prev = magnitude_case(d, route, target)
    r64 = ref_step(_f64(W), d, (_f64(state[0]), _f64(state[1]), state[2]), prev, _f64(statics), False)
    got = {mode: dev_step(_model(monkeypatch, mode, d, W), state, prev, _cuda(statics), False) for mode in MODES}
    for mode in ("f16+f8x2", "f16x3"):
        b_tc, b_simt = step_bounds(mode, r64, state), step_bounds("simt", r64, state)
        ratio = {q: bound_ratio(got[mode][q], got["simt"][q], b_tc[q] + b_simt[q]) for q in QUANTITIES}
        print(f"DECODER-F64 att~{target:g} via {route}: {mode} vs simt / bound "
              + " ".join(f"{q} {ratio[q]:.3f}" for q in QUANTITIES))
        for q in QUANTITIES:
            assert ratio[q] <= 1.0, (route, target, mode, q, ratio[q])


# ----------------------------------------------------------------------------- 3. whole decodes
def _decode_inputs(d, b, seed):
    return O.synth_inputs(b, 30, 8, 20, d.det_feat_size, seed=seed, vocab_size=d.vocab_size, n_det_range=(5, 30),
                          real_slots=(2, 8), verb_slots=(1,), verb_vocab_id=17)


def _check_beam(tag, d, W, m, statics, k, trace):
    from gpu_common import device_beam
    (w, g), (lw, lg), hist, extra = device_beam(m, _cuda(statics), [3, -1], k, 1, True, True, trace=trace)
    so, sg = (extra["step_out"], extra["step_gate"]) if trace else (None, None)
    for label, WW, st in (("float64", _f64(W), _f64(statics)), ("float32", W, statics)):
        v, o_outs, o_lps = verify_device_beam(WW, d, st, [3, -1], k, hist, True, True, None, so, sg)
        print(f"DECODER-F64 {tag} vs {label} oracle: {v.summary()}")
        assert not v.violations, (tag, label, v.violations[:3])
        assert v.max_out_rel <= 1.0 and v.max_gate_rel <= 1.0, (tag, label, v.summary())
        check_returned_beams(f"{tag} {label}", d, hist, 1, (w, g, lw, lg), o_outs, o_lps)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("trace", [True, False], ids=["trace", "fused-head"])
@pytest.mark.parametrize("d", [FULL, ODD_V], ids=["V10000", "V97"])
def test_beam_search_at_trained_like_parameters(monkeypatch, mode, trace, d):
    """V = 97 leaves 15 pad columns in the last 16-column chunk of the fused head's per-chunk softmax records."""
    W = trained_like(d, seed=21)
    m = _model(monkeypatch, mode, d, W)
    tag = f"beam V={d.vocab_size} b=8 k=3 {'trace' if trace else 'fused head'}"
    _check_beam(tag, d, W, m, _decode_inputs(d, 8, 61), 3, trace)


STACKED = O.Dims(seq_len=6)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_stacked_beam_search_at_trained_like_parameters(monkeypatch, mode):
    """128 captions x beam 5 = 640 rows: every step GEMM on the CTA-pair kernel."""
    d = STACKED
    W = trained_like(d, seed=22)
    m = _model(monkeypatch, mode, d, W)
    _check_beam("stacked beam b=128 k=5", d, W, m, _decode_inputs(d, 128, 62), 5, False)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_forward_at_trained_like_parameters(monkeypatch, mode):
    d = FULL
    W = trained_like(d, seed=23)
    m = _model(monkeypatch, mode, d, W)
    det, ds, _ = _decode_inputs(d, 8, 63)
    caps = torch.randint(0, d.vocab_size, (8, d.seq_len), generator=torch.Generator().manual_seed(5))
    ctrl = torch.stack([ds[:, min(t // 2, ds.size(1) - 1)] for t in range(d.seq_len)], 1).contiguous()
    out, gate = m((det.to(DEV),), (caps.to(DEV), ctrl.to(DEV)))
    torch.cuda.synchronize()
    with torch.no_grad():
        r64 = O.forward_teacher(_f64(W), d, (det.double(),), (caps, ctrl.double()))
        r32 = O.forward_teacher(W, d, (det,), (caps, ctrl))
    for got, ref, name in ((out.cpu(), r64[0], "out"), (gate.cpu(), r64[1], "gate")):
        assert rel_close(r32[0 if name == "out" else 1], ref, REL, ABS), (mode, name, "fp32 oracle")
        assert rel_close(got, ref, REL, ABS), (mode, name)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
def test_greedy_at_trained_like_parameters(monkeypatch, mode):
    """Each device pick, replayed through the float64 oracle, is an arg-max up to the tie band; the float32 oracle's own
    greedy decode picks within the same band."""
    d = FULL
    W = trained_like(d, seed=24)
    m = _model(monkeypatch, mode, d, W)
    det, ds, _ = _decode_inputs(d, 8, 64)
    words, gates = m.test(det.to(DEV), ds.to(DEV))
    torch.cuda.synchronize()
    W64, st64 = _f64(W), (det.double(), ds.double())
    o32_w, o32_g = O.greedy_test(W, d, (det, ds))
    for label, pw_all, pg_all in (("device", words.cpu(), gates.cpu()), ("float32 oracle", o32_w, o32_g)):
        state, prev = O.init_state(d, det.size(0), torch.float64), None
        with torch.no_grad():
            for t in range(d.seq_len):
                (out, gate), state = O.decoder_step(W64, d, t, state, prev, st64, None, "feedback")
                pw, pg = pw_all[:, t], pg_all[:, t]
                band = 2e-3 + 1e-4 * out.max(1).values.abs()
                assert bool((out.gather(1, pw[:, None]).squeeze(1) >= out.max(1).values - band).all()), (mode, label, t)
                assert bool((gate.gather(1, pg[:, None]).squeeze(1) >= gate.max(1).values - 2e-3).all()), (mode, label, t)
                prev = (pw, pg)


# ----------------------------------------------------------------------------- 4. CPU: the float64 oracle
def test_float64_oracle_at_trained_like_parameters():
    """The float64 oracle reproduces the reference's golden vectors (zero-bias init) and, at trained-like parameters,
    agrees with the float32 oracle well inside the bounds above on a small model."""
    fx = load_golden("small_a.pt")
    d, W = fx["dims_obj"], fx["weights"]
    det, ds, vg = fx["det"], fx["det_seqs"], fx["verbs_gt"]
    c = fx["cases"]["step_v"]
    with torch.no_grad():
        st = O.init_state(d, det.size(0), torch.float64)
        (o0, g0), st = O.decoder_step(_f64(W), d, 0, st, None, _f64((det, ds, vg)), None, "feedback", use_verbs=True,
                                      gt=True)
        (o1, g1), st = O.decoder_step(_f64(W), d, 1, st, (c["prev_word"], c["prev_gate"]), _f64((det, ds, vg)), None,
                                      "feedback", use_verbs=True, gt=True)
    for got, ref in ((o0, c["out0"]), (g0, c["gate0"]), (o1, c["out1"]), (g1, c["gate1"]),
                     (st[0][0], c["h1"]), (st[0][1], c["c1"]), (st[1][0], c["h2"]), (st[1][1], c["c2"])):
        assert rel_close(got, ref, 1e-5, 1e-6)
    # trained-like parameters: every bias non-zero, forget gates offset, and the float32 oracle inside every bound
    Wt = trained_like(d, seed=3)
    for k in Wt:
        if k.endswith("bias") or "bias_" in k:
            assert float(Wt[k].abs().min()) > 0, k
    assert float(Wt["out_fc.bias"].mean()) < -29
    statics, state, prev = step_inputs(d, 9, 6, seed=5, L=4, D=9, verbs=True)
    r64 = ref_step(_f64(Wt), d, (_f64(state[0]), _f64(state[1]), state[2]), prev, _f64(statics), True)
    r32 = ref_step(Wt, d, state, prev, statics, True)
    bounds = step_bounds("simt", r64, state)
    for q in QUANTITIES:
        assert bound_ratio(r32[q], r64[q], bounds[q]) <= 1.0, q
    # a dropped bias term moves the step far outside the bounds
    Wd = dict(Wt)
    Wd["lstm_cell_2.bias_hh"] = torch.zeros_like(Wt["lstm_cell_2.bias_hh"])
    rd = ref_step(Wd, d, state, prev, statics, True)
    assert bound_ratio(rd["h2"], r64["h2"], step_bounds("f16+f8x2", r64, state)["h2"]) > 10
