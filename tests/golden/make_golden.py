"""Generate golden vectors from the UNMODIFIED reference (a checkout of the original project).

    VSR_REFERENCE_ROOT=<checkout> python tests/golden/make_golden.py

Imports $VSR_REFERENCE_ROOT/models, runs the reference's own ``beam_search_v`` /
``beam_search`` / ``forward`` / ``test`` / ``step_v`` on seeded synthetic inputs and
stores inputs + outputs as small ``.pt`` fixtures beside this script:

  small_a.pt   default flags, tiny dims (weights + inputs stored verbatim)
  small_b.pt   h2_first_lstm=False, img_second_lstm=True, tiny dims
  full_cfg1.pt BASELINE config 1 at full model size: outputs only, plus float64
               checksums of the seeded weights/inputs so a box whose RNG stream
               differs can detect it and skip instead of failing.

These files are the parity pin for oracle/vsr_oracle.py (the reference has no tests
or golden vectors of its own: SURVEY.md §4).
"""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import refload  # noqa: E402
from oracle import vsr_oracle as O  # noqa: E402
from oracle.ssp_oracle import checksum  # noqa: E402


def run_small(path, dims: O.Dims, seed_w, seed_x):
    table = O.synth_verb_table(40, dims.vocab_size, seed=7)
    m = refload.build_reference_model(dims.asdict(), seed=seed_w, verb_table=table)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    b, D, L, R, Fd = 6, 12, 10, 20, dims.det_feat_size
    det, ds, verbs_gt = O.synth_inputs(b, D, L, R, Fd, seed=seed_x, vocab_size=dims.vocab_size,
                                       n_det_range=(5, 12), verb_slots=(2,), verb_vocab_id=17)
    verbs_tab = verbs_gt.clone()
    g = torch.Generator().manual_seed(seed_x + 1)
    vmask = verbs_tab != -1
    verbs_tab[vmask] = torch.randint(0, 44, (int(vmask.sum()),), generator=g).double()  # some ids absent
    verbs_tab[0, 4] = 3.0                                                                # a second verb slot
    T = dims.seq_len
    caps = torch.randint(0, dims.vocab_size, (b, T), generator=g)
    ctrl = torch.zeros((b, T, R, Fd))
    for i in range(b):
        for t in range(T):
            ctrl[i, t] = ds[i, min(t // 2, L - 1)]
    fx = {"dims": dims.asdict(), "weights": sd, "verb_table": table,
          "det": det, "det_seqs": ds, "verbs_gt": verbs_gt, "verbs_tab": verbs_tab,
          "captions": caps, "ctrl_rule": "ctrl[i,t] = det_seqs[i, min(t//2, L-1)]", "cases": {}}
    with torch.no_grad():
        o, lp = m.beam_search_v((det, ds, verbs_gt), [3, -1], 3, 1, gt=True)
        fx["cases"]["bsv_gt_k3"] = {"eos": [3, -1], "beam": 3, "out_size": 1, "out": o, "lp": lp}
        o, lp = m.beam_search_v((det, ds, verbs_tab), [3, -1], 5, 1, gt=False)
        fx["cases"]["bsv_tab_k5"] = {"eos": [3, -1], "beam": 5, "out_size": 1, "out": o, "lp": lp}
        o, lp = m.beam_search((det, ds), [3, 1], 4, 2)
        fx["cases"]["bs_freeze_k4"] = {"eos": [3, 1], "beam": 4, "out_size": 2, "out": o, "lp": lp}
        o, lp = m.beam_search_v((det[:1], ds[:1], verbs_gt[:1]), [3, -1], 3, 1, gt=True)
        fx["cases"]["bsv_gt_b1"] = {"eos": [3, -1], "beam": 3, "out_size": 1, "out": o, "lp": lp}
        out, gate = m((det,), (caps, ctrl))
        fx["cases"]["forward"] = {"out": out, "gate": gate}
        w, gts = m.test(det, ds)
        fx["cases"]["greedy"] = {"words": w, "gates": gts}
        # two consecutive feedback steps of step_v from a non-trivial state
        st = m.init_state(b, "cpu")
        (o0, g0), st = m.step_v(0, st, None, (det, ds, verbs_gt), None, mode="feedback", gt=True)
        pw, pg = o0.argmax(-1), torch.ones(b, dtype=torch.long)
        (o1, g1), st = m.step_v(1, st, [pw, pg], (det, ds, verbs_gt), None, mode="feedback", gt=True)
        fx["cases"]["step_v"] = {"out0": o0, "gate0": g0, "prev_word": pw, "prev_gate": pg,
                                 "out1": o1, "gate1": g1,
                                 "h1": st[0][0], "c1": st[0][1], "h2": st[1][0], "c2": st[1][1], "ptr": st[2]}
    torch.save(fx, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


def run_full_cfg1(path):
    dims = O.Dims()
    m = refload.build_reference_model(dims.asdict(), seed=1234)
    sd = m.state_dict()
    det, ds, verbs = O.synth_inputs(8, 20, 10, 20, 2048, seed=1001, vocab_size=dims.vocab_size,
                                    verb_slots=(2,), verb_vocab_id=17, real_slots=(6, 6))
    fx = {"dims": dims.asdict(), "seed_w": 1234,
          "synth": dict(b=8, D=20, L=10, R=20, Fd=2048, seed=1001, vocab_size=dims.vocab_size,
                        verb_slots=(2,), verb_vocab_id=17, real_slots=(6, 6)),
          "weight_checksums": {k: checksum(v) for k, v in sd.items()},
          "input_checksums": {"det": checksum(det), "det_seqs": checksum(ds), "verbs": checksum(verbs)},
          "cases": {}}
    with torch.no_grad():
        o, lp = m.beam_search_v((det, ds, verbs), [3, -1], 3, 1, gt=True)
        fx["cases"]["bsv_gt_k3"] = {"eos": [3, -1], "beam": 3, "out_size": 1, "out": o, "lp": lp}
        # sharpened variant (SURVEY §7): out_fc.weight *= 100 makes most beam decisions decisive
        m.out_fc.weight.mul_(100.0)
        o, lp = m.beam_search_v((det, ds, verbs), [3, -1], 3, 1, gt=True)
        fx["cases"]["bsv_gt_k3_sharp100"] = {"eos": [3, -1], "beam": 3, "out_size": 1, "out": o, "lp": lp}
    torch.save(fx, path)
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    assert refload.available(), "set VSR_REFERENCE_ROOT to a checkout of the original project"
    small = dict(seq_len=20, vocab_size=157, bos_idx=2, det_feat_size=96, input_encoding_size=36,
                 rnn_size=50, att_size=20)
    run_small(os.path.join(HERE, "small_a.pt"), O.Dims(**small), seed_w=1234, seed_x=1001)
    run_small(os.path.join(HERE, "small_b.pt"),
              O.Dims(**small, h2_first_lstm=False, img_second_lstm=True), seed_w=4321, seed_x=1002)
    run_full_cfg1(os.path.join(HERE, "full_cfg1.pt"))
