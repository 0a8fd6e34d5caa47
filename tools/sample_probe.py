"""Sampling decode with several draws per caption (vsr_sample_ex) on the benchmarked workload's inputs (config 2:
D = 50, L = 10, R = 20, F = 2048, V = 10000, T = 20, raw weights of torch.manual_seed(1234), bench.py's seeds 1002..),
at 100 and 1000 captions, 5 captions' worth of rows per caption in every arm:

  a. sample_rl on the captions repeated 5x (repeat_interleave of det / det_seqs: 5x the prologue and the inputs)
  b. sample_rl(n=5)
  c. sample_rl(n=5, top_k=40)
  d. sample_rl(n=5, top_p=0.9)
  e. sample_rl(n=5, temperature=0.7, top_p=0.9)
  f. sample_v(n=5, gt=True, top_p=0.9)
  g. beam_search_v, beam 5 (graph replay), for context: the same number of rows per step

All arms run in one process and alternate round by round (the order rotates every round); ms per call by CUDA events,
median [min, max] over `--rounds` rounds.  Then, in separate rounds with the phase profiler on (no graph replay), the
pick phase (`beam_select`: k_sample_pick, or the beam selection) and the whole decode, per call.

    python tools/sample_probe.py [--rounds 7] [--out profiles/sample_probe_b200.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "vsr-guided-cic_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from tools.synth import synth_inputs  # noqa: E402

EOS = [3, -1]
N = 5


def batch(b):
    parts = [synth_inputs(100, 50, 10, 20, 2048, seed=1002 + i, vocab_size=10000, n_det_range=(10, 50),
                          verb_slots=(2,), verb_vocab_id=17) for i in range(b // 100)]
    return tuple(torch.cat(x, 0) for x in zip(*parts))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_probe: needs a CUDA device")
    from models import ControllableCaptioningModel
    dev = "cuda:0"
    torch.manual_seed(1234)
    model = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()
    result = {"card": card(), "rounds": args.rounds, "draws_per_caption": N,
              "workload": "config2 inputs, D=50 L=10 R=20 F=2048 V=10000 T=20, raw weights (torch.manual_seed(1234))"}
    sizes = {100: 5, 1000: 2}
    for b, calls in sizes.items():
        det, ds, verbs = (t.to(dev) for t in batch(b))
        det5, ds5 = det.repeat_interleave(N, 0), ds.repeat_interleave(N, 0)
        arms = {
            "a_repeat5_sample_rl": lambda: model.sample_rl(det5, ds5, seed=1),
            "b_n5": lambda: model.sample_rl(det, ds, seed=1, n=N),
            "c_n5_topk40": lambda: model.sample_rl(det, ds, seed=1, n=N, top_k=40),
            "d_n5_topp0.9": lambda: model.sample_rl(det, ds, seed=1, n=N, top_p=0.9),
            "e_n5_t0.7_topp0.9": lambda: model.sample_rl(det, ds, seed=1, n=N, temperature=0.7, top_p=0.9),
            "f_sample_v_n5_gt_topp0.9": lambda: model.sample_v((det, ds, verbs), n=N, gt=True, top_p=0.9, seed=1),
            "g_beam_search_v_k5": lambda: model.beam_search_v((det, ds, verbs), EOS, N, 1, gt=True),
        }

        def run(fn, k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k

        for fn in arms.values():                          # warm: every shape, eager + graph capture + replay
            run(fn, 3)
        names = list(arms)
        ms = {n: [] for n in names}
        for r in range(args.rounds):
            rot = names[r % len(names):] + names[:r % len(names)]
            for n in rot:
                ms[n].append(run(arms[n], calls))
        # phase profiler: separate rounds (events around every launch, no graph replay)
        eng = model._engine()
        eng.set_profiling(True)
        pick = {n: [] for n in names}
        total = {n: [] for n in names}
        for r in range(args.rounds):
            rot = names[r % len(names):] + names[:r % len(names)]
            for n in rot:
                arms[n]()
                torch.cuda.synchronize()
                pt = {name: t for name, t, _ in eng.phase_times()}
                pick[n].append(pt["beam_select"])
                total[n].append(sum(pt.values()))
        eng.set_profiling(False)
        rec = {"calls_per_round": calls, "rows_per_step": b * N}
        for n in names:
            rec[n] = {"ms_per_call": summary(ms[n]), "profiled_pick_ms": summary(pick[n]),
                      "profiled_phases_ms": summary(total[n])}
            print(json.dumps({"captions": b, "arm": n, "ms_per_call": rec[n]["ms_per_call"]["median"],
                              "pick_ms": rec[n]["profiled_pick_ms"]["median"],
                              "phases_ms": rec[n]["profiled_phases_ms"]["median"]}), flush=True)
        result[str(b)] = rec
        del det5, ds5, det, ds, verbs
        torch.cuda.empty_cache()
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
