"""Live check of the oracle against the UNMODIFIED reference (only where VSR_REFERENCE_ROOT names a
checkout of the original project; skipped elsewhere).  test_oracle_golden.py keeps the comparison
against vectors the reference produced, without it."""
import pytest
import torch

import refload
from oracle import vsr_oracle as O

pytestmark = pytest.mark.skipif(not refload.available(),
                                reason="the original project is not present (set VSR_REFERENCE_ROOT to its checkout)")


@pytest.mark.parametrize("flags", [(True, False), (False, False), (True, True)])
def test_init_and_beam_search_bit_exact(flags):
    d = O.Dims(seq_len=12, vocab_size=131, bos_idx=2, det_feat_size=64, input_encoding_size=28,
               rnn_size=34, att_size=12, h2_first_lstm=flags[0], img_second_lstm=flags[1])
    table = O.synth_verb_table(30, d.vocab_size, seed=3)
    m = refload.build_reference_model(d.asdict(), seed=99, verb_table=table)
    W = O.init_weights(d, seed=99)
    sd = m.state_dict()
    assert list(sd.keys()) == list(W.keys()) == list(O.param_shapes(d).keys())
    for k in sd:
        assert torch.equal(sd[k], W[k]), k
    det, ds, verbs = O.synth_inputs(5, 9, 6, 7, 64, seed=5, vocab_size=131, n_det_range=(3, 9),
                                    real_slots=(3, 6), verb_slots=(1, 3), verb_id_range=(0, 33))
    with torch.no_grad():
        for gt in (True, False):
            v = verbs.clone()
            if gt:
                v[v != -1] = v[v != -1].remainder(131)
            ro, rl = m.beam_search_v((det, ds, v), [3, -1], 4, 2, gt=gt)
            oo, ol = O.beam_search(W, d, (det, ds, v), [3, -1], 4, 2, use_verbs=True, gt=gt, verb_table=table)
            for a, b in zip(ro + rl, oo + ol):
                assert torch.equal(a, b)
        ro, rl = m.beam_search((det, ds), [3, 0], 3, 3)
        oo, ol = O.beam_search(W, d, (det, ds), [3, 0], 3, 3)
        for a, b in zip(ro + rl, oo + ol):
            assert torch.equal(a, b)
