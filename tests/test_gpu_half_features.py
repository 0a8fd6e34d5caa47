"""Half-precision region features (fp16 / bf16) through every decode driver.

Widening fp16 or bf16 to fp32 is exact, and every kernel that reads features widens each value as it loads it and then
does the fp32 path's arithmetic in the same order.  So a decode of half-precision inputs x must equal, bit for bit, the
decode of x.float() on the same model; the fp32 path is the one the parity suite pins to the oracle.  Every comparison
here is torch.equal, with no tolerance.

GPU tests are marked one by one: the CPU-only cases at the end run without a device."""
import os
import re
import subprocess

import pytest
import torch

from oracle import vsr_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"
HALF = [torch.float16, torch.bfloat16]


def _cuda(*ts):
    return tuple(t.to(DEV) for t in ts)


def _as(dtype, det, feats, verbs=None):
    """(det, feats[, verbs]) on the device with the features in `dtype`."""
    out = (det.to(DEV, dtype), feats.to(DEV, dtype) if feats.is_floating_point() else feats.to(DEV))
    return out if verbs is None else out + (verbs.to(DEV),)


def _up(statics):
    """The fp32 upcast of the half-precision features (index tensors and verbs unchanged)."""
    return tuple(t.float() if t.dtype in HALF else t for t in statics)


def _equal(a, b, what):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), what
        for k in a:
            _equal(a[k], b[k], f"{what}[{k}]")
    elif isinstance(a, (tuple, list)):
        assert len(a) == len(b), what
        for i, (x, y) in enumerate(zip(a, b)):
            _equal(x, y, f"{what}[{i}]")
    else:
        assert a.dtype == b.dtype and a.shape == b.shape, what
        assert torch.equal(a, b), what


def _config2_inputs(b=100, seed=1002):
    return O.synth_inputs(b, 50, 10, 20, 2048, seed=seed, vocab_size=10000, n_det_range=(10, 50), verb_slots=(2,),
                          verb_vocab_id=17)


def _model(d, seed=1234, sharpen=None):
    from gpu_common import make_model
    W = O.init_weights(d, seed=seed)
    if sharpen:
        W["out_fc.weight"] = W["out_fc.weight"] * sharpen
    return make_model(d, W)


@pytest.fixture(scope="module")
def cfg2():
    """Config 2 with the raw init_weights(1234) model: the benchmarked workload."""
    return _model(O.Dims())


def _beam(m, statics, k=5, out_size=1, indexed=False, attention=False):
    fn = m.beam_search_v_indexed if indexed else m.beam_search_v
    res = fn(statics, [3, -1], k, out_size, gt=True, return_attention=attention)
    hist = m._eng.history()
    torch.cuda.synchronize()
    return res, [h.clone() for h in hist]


# ----------------------------------------------------------------------------- 1. materialised slot tiles
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_beam_search_v_equals_upcast(cfg2, dtype):
    """Config 2 raw, b = 100, beam 5: words, gates, both log-prob tensors and the beam history; then with the
    attention returned, and with out_size 3."""
    det, ds, verbs = _config2_inputs()
    half = _as(dtype, det, ds, verbs)
    up = _up(half)
    for out_size, attention in ((1, False), (1, True), (3, False)):
        got, hist = _beam(cfg2, half, out_size=out_size, attention=attention)
        want, hist_up = _beam(cfg2, up, out_size=out_size, attention=attention)
        tag = f"{dtype} out_size={out_size} attention={attention}"
        _equal(got, want, tag)
        _equal(hist, hist_up, tag + " history")


# ----------------------------------------------------------------------------- 2. index form
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("shared_image", [False, True])
def test_beam_search_v_indexed_equals_upcast(cfg2, dtype, shared_image):
    """Dense (b, D, F) detections and one stride-0 shared image.  The -2 slots read the fp32 image mean row, so one
    slot tile mixes half-precision detection rows with an fp32 row."""
    det, idx, verbs = O.synth_inputs_indexed(100, 50, 10, 20, 2048, seed=1006, n_det_range=(10, 50))
    if shared_image:
        idx = idx.clamp(max=int((det[0].sum(-1) != 0).sum()) - 1)
        d_h = det[:1].to(DEV, dtype).expand(100, 50, 2048)
        d_up = d_h[:1].float().expand(100, 50, 2048)        # the same stride-0 layout in fp32
    else:
        d_h = det.to(DEV, dtype)
        d_up = d_h.float()
    # tiles that hold the mean row next to detection rows
    idx[:, 3, 0] = -2
    assert bool(((idx == -2).any(-1) & (idx >= 0).any(-1)).any())
    idx, verbs = idx.to(DEV), verbs.to(DEV)
    got, hist = _beam(cfg2, (d_h, idx, verbs), indexed=True, attention=True)
    want, hist_up = _beam(cfg2, (d_up, idx, verbs), indexed=True, attention=True)
    _equal(got, want, f"{dtype} shared={shared_image}")
    _equal(hist, hist_up, f"{dtype} shared={shared_image} history")


# ----------------------------------------------------------------------------- 3. the other drivers
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_forward_greedy_sample_and_step_equal_upcast(cfg2, dtype):
    m = cfg2
    b = 40
    det, ds, verbs = O.synth_inputs(b, 100, 10, 20, 2048, seed=1005, vocab_size=10000, n_det_range=(10, 100))
    caps = torch.randint(0, 10000, (b, 20), generator=torch.Generator().manual_seed(7)).to(DEV)
    ctrl = torch.stack([ds[:, min(t // 2, 9)] for t in range(20)], 1).contiguous()
    det_h, ctrl_h = det.to(DEV, dtype), ctrl.to(DEV, dtype)
    # teacher-forced forward (out and gate)
    got = m((det_h,), (caps, ctrl_h))
    want = m((det_h.float(),), (caps, ctrl_h.float()))
    _equal(got, want, f"{dtype} forward")
    half = _as(dtype, det, ds, verbs)
    up = _up(half)
    # greedy
    _equal(m.test(*half[:2]), m.test(*up[:2]), f"{dtype} greedy")
    # sampling with a fixed seed
    _equal(m.sample_rl(*half[:2], seed=123), m.sample_rl(*up[:2], seed=123), f"{dtype} sample_rl")
    # single steps of step_v with a verb table (gt=False)
    m._eng.set_verb_table({"17": [5, 9, 21]})
    try:
        g = torch.Generator().manual_seed(3)
        prev = (torch.randint(0, 10000, (b,), generator=g).to(DEV), torch.randint(0, 2, (b,), generator=g).to(DEV))
        outs = []
        for statics in (half, up):
            state = m.init_state(b, DEV)
            r0, state = m.step_v(0, state, None, statics, None, mode="feedback", gt=False)
            r1, state = m.step_v(1, state, prev, statics, None, mode="feedback", gt=False)
            outs.append((r0, r1, state))
        _equal(outs[0], outs[1], f"{dtype} step_v")
    finally:
        m._eng.set_verb_table({})


# ----------------------------------------------------------------------------- 4. caption independence, CTA pairs
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_stacked_1150_row_decode_equals_upcast(cfg2, dtype):
    """230 captions x beam 5 = 1150 rows: the step GEMMs run on the CTA-pair kernels."""
    a = _config2_inputs()
    extra = _config2_inputs(130, seed=1003)
    det, ds, verbs = (torch.cat([x, y], 0) for x, y in zip(a, extra))
    half = _as(dtype, det, ds, verbs)
    got, hist = _beam(cfg2, half)
    want, hist_up = _beam(cfg2, _up(half))
    _equal(got, want, f"{dtype} 1150 rows")
    _equal(hist, hist_up, f"{dtype} 1150 rows history")


# ----------------------------------------------------------------------------- 5. GEMM modes
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_f16x3_mode_equals_upcast(monkeypatch, dtype):
    monkeypatch.setenv("VSRDEC_GEMM", "f16x3")       # read when the handle is created
    m = _model(O.Dims(), sharpen=100.0)
    det, ds, verbs = _config2_inputs(b=24)
    half = _as(dtype, det, ds, verbs)
    got, hist = _beam(m, half)
    assert m._eng.gemm_kind() == "tcgen05-f16x3"
    want, hist_up = _beam(m, _up(half))
    _equal(got, want, f"{dtype} f16x3")
    _equal(hist, hist_up, f"{dtype} f16x3 history")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_simt_mode_rejects_half_features(monkeypatch, dtype):
    from vsrdec import VsrError
    monkeypatch.setenv("VSRDEC_GEMM", "simt")
    d = O.Dims(seq_len=6, vocab_size=97, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    m = _model(d)
    det, ds, verbs = O.synth_inputs(5, 9, 5, 6, 64, seed=21, vocab_size=97, n_det_range=(3, 9), real_slots=(2, 5),
                                    verb_slots=(1,), verb_vocab_id=11)
    m.beam_search_v(_cuda(det, ds, verbs), [3, -1], 3, 1, gt=True)        # fp32 still runs
    assert m._eng.gemm_kind() == "simt-fp32"
    with pytest.raises(VsrError, match="fp32 FFMA twin"):
        m.beam_search_v(_as(dtype, det, ds, verbs), [3, -1], 3, 1, gt=True)


# ----------------------------------------------------------------------------- 6. graph cache
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_graph_cache_keys_on_the_feature_dtype(dtype):
    """fp32, then half precision in tensors that start at the SAME device addresses with the same shapes, then fp32
    again; each twice, so that the second call replays the prologue's and the steps' graphs.  Every result equals a
    fresh decode of its own dtype.  Then new half-precision data in the same buffers is picked up on replay."""
    m = _model(O.Dims(), sharpen=100.0)
    b = 16
    det, ds, verbs = _config2_inputs(b=b)
    det2, ds2, _ = _config2_inputs(b=b, seed=77)
    nd, ns = det.numel(), ds.numel()
    buf_d = torch.zeros(nd * 4, dtype=torch.uint8, device=DEV)
    buf_s = torch.zeros(ns * 4, dtype=torch.uint8, device=DEV)
    v = verbs.to(DEV)

    def views(dt):
        n = torch.finfo(dt).bits // 8
        return buf_d[:nd * n].view(dt).view(det.shape), buf_s[:ns * n].view(dt).view(ds.shape)

    def fresh(dt, d_, s_):
        # separate tensors at other addresses: an eager decode, never a replay of the shared buffers' graphs
        got, hist = _beam(m, (d_.to(DEV, dt).clone(), s_.to(DEV, dt).clone(), v))
        return got, hist

    refs = {dt: fresh(dt, det, ds) for dt in (torch.float32, dtype)}
    for dt in (torch.float32, dtype, torch.float32):
        dv, sv = views(dt)
        assert dv.data_ptr() == buf_d.data_ptr() and sv.data_ptr() == buf_s.data_ptr()
        dv.copy_(det.to(dt)), sv.copy_(ds.to(dt))
        for call in range(2):
            got, hist = _beam(m, (dv, sv, v))
            _equal(got, refs[dt][0], f"{dt} call {call}")
            _equal(hist, refs[dt][1], f"{dt} call {call} history")
    # new data written into the same half-precision buffers
    want = fresh(dtype, det2, ds2)
    dv, sv = views(dtype)
    dv.copy_(det2.to(dtype)), sv.copy_(ds2.to(dtype))
    for call in range(2):
        got, hist = _beam(m, (dv, sv, v))
        _equal(got, want[0], f"{dtype} new data call {call}")
        _equal(hist, want[1], f"{dtype} new data call {call} history")


# ----------------------------------------------------------------------------- 7. feature width
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_feature_width_4_mod_8_equals_upcast(dtype):
    """F = 132: a half-precision row is only 8-byte aligned, every other row starts mid 16-byte word."""
    d = O.Dims(seq_len=8, bos_idx=2, vocab_size=513, det_feat_size=132, input_encoding_size=64, rnn_size=130,
               att_size=36, h2_first_lstm=False)
    m = _model(d, seed=5, sharpen=30.0)
    det, ds, verbs = O.synth_inputs(7, 9, 5, 6, 132, seed=21, vocab_size=513, n_det_range=(3, 9), real_slots=(2, 5),
                                    verb_slots=(1,), verb_vocab_id=11)
    half = _as(dtype, det, ds, verbs)
    got, hist = _beam(m, half, k=4, out_size=2, attention=True)
    want, hist_up = _beam(m, _up(half), k=4, out_size=2, attention=True)
    _equal(got, want, f"{dtype} F=132")
    _equal(hist, hist_up, f"{dtype} F=132 history")
    det_i, idx, verbs_i = O.synth_inputs_indexed(7, 9, 5, 6, 132, seed=22, n_det_range=(3, 9), real_slots=(2, 5),
                                                 verb_slots=(1,), verb_vocab_id=11)
    dh = det_i.to(DEV, dtype)
    got, _ = _beam(m, (dh, idx.to(DEV), verbs_i.to(DEV)), k=4, indexed=True)
    want, _ = _beam(m, (dh.float(), idx.to(DEV), verbs_i.to(DEV)), k=4, indexed=True)
    _equal(got, want, f"{dtype} F=132 indexed")


# ----------------------------------------------------------------------------- 8. pipeline
@pytest.mark.gpu
@pytest.mark.parametrize("stack", [1, 3])
def test_decode_pipeline_takes_pinned_fp16_batches(stack):
    from vsrdec import DecodePipeline
    from gpu_common import make_model
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    W["out_fc.weight"] = W["out_fc.weight"] * 100.0
    models = [make_model(d, W), make_model(d, W)]
    batches = []
    for i in range(5):
        det, ds, verbs = O.synth_inputs(12, 50, 10, 20, 2048, seed=3000 + i, vocab_size=d.vocab_size,
                                        n_det_range=(10, 50), verb_slots=(2,), verb_vocab_id=17)
        batches.append((det.half(), ds.half(), verbs))
    pinned = [tuple(t.pin_memory() for t in b_) for b_ in batches]
    pipe = DecodePipeline(models, [3, -1], 5, 1, gt=True, buffers=4, stack=stack)
    got = list(pipe.run(iter(pinned)))
    assert len(got) == len(batches)
    for i, b_ in enumerate(batches):
        (w, g), (lw, lg) = models[0].beam_search_v(_up(_cuda(*b_)), [3, -1], 5, 1, gt=True)
        torch.cuda.synchronize()
        _equal(tuple(got[i]), (w.cpu(), g.cpu(), lw.cpu(), lg.cpu()), f"batch {i}")


# ----------------------------------------------------------------------------- 9. errors
@pytest.mark.gpu
def test_feature_dtype_errors():
    from vsrdec import VsrError
    d = O.Dims(seq_len=6, vocab_size=97, det_feat_size=64, input_encoding_size=30, rnn_size=33, att_size=12)
    m = _model(d)
    det, ds, verbs = O.synth_inputs(5, 9, 5, 6, 64, seed=21, vocab_size=97, n_det_range=(3, 9), real_slots=(2, 5),
                                    verb_slots=(1,), verb_vocab_id=11)
    with pytest.raises(VsrError, match="share one dtype"):
        m.beam_search_v((det.to(DEV, torch.float16), ds.to(DEV), verbs.to(DEV)), [3, -1], 3, 1, gt=True)
    with pytest.raises(VsrError, match="float64"):
        m.beam_search_v(_as(torch.float64, det, ds, verbs), [3, -1], 3, 1, gt=True)
    with pytest.raises(VsrError, match="float64"):
        m.beam_search_v_indexed((det.to(DEV, torch.float64), torch.zeros((5, 6, 6), dtype=torch.int32, device=DEV)),
                                [3, -1], 3, 1)
    eng = m._engine()
    dh, sh = det.to(DEV, torch.float16), ds.to(DEV, torch.float16)
    lib = eng.lib
    rc = lib.vsr_prologue_ex(eng.handle, dh.data_ptr(), 9 * 64, 9, sh.data_ptr(), 5, 6, 6, 7, None, 0, None)
    assert rc == -1 and b"feat_dtype=7" in lib.vsr_last_error()                          # VSR_EINVAL
    idx = torch.zeros((5, 6, 6), dtype=torch.int32, device=DEV)
    rc = lib.vsr_prologue_indexed_ex(eng.handle, dh.data_ptr(), 9 * 64, 9, idx.data_ptr(), 5, 6, 6, 7, None, 0, None)
    assert rc == -1
    # half-precision rows need 8-byte alignment, not 16 (b = 4 of the 5 images: the shifted reads stay inside det)
    assert lib.vsr_prologue_ex(eng.handle, dh.data_ptr() + 8, 9 * 64, 9, sh.data_ptr(), 4, 6, 6, 3, None, 0, None) == 0
    assert lib.vsr_prologue_ex(eng.handle, dh.data_ptr() + 4, 9 * 64, 9, sh.data_ptr(), 4, 6, 6, 3, None, 0, None) == -1
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------- 10. CPU-only
def _header():
    return open(os.path.join(ROOT, "include", "vsrdec.h")).read()


def test_header_declares_the_half_precision_prologues():
    src = re.sub(r"/\*.*?\*/", "", _header(), flags=re.S)
    assert {"vsr_prologue_ex", "vsr_prologue_indexed_ex"} <= set(re.findall(r"\b(vsr_[a-z_0-9]+)\s*\(", src))
    tags = dict(re.findall(r"#define\s+(VSR_DT_[A-Z0-9]+)\s+(\d+)", src))
    assert tags.get("VSR_DT_F16") == "3" and tags.get("VSR_DT_BF16") == "4" and tags.get("VSR_DT_F32") == "1"
    import vsrdec
    assert {"vsr_prologue_ex", "vsr_prologue_indexed_ex"} <= set(vsrdec.EXPORTED_SYMBOLS)


def test_library_exports_the_half_precision_prologues():
    import vsrdec
    path = vsrdec.library_path()
    if not os.path.isfile(path):
        pytest.skip("libvsrdec.so is not built")
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True).stdout
    assert {"vsr_prologue_ex", "vsr_prologue_indexed_ex"} <= set(re.findall(r" T (vsr_[a-z_0-9]+)", out))
