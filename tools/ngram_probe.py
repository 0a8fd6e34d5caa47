"""Cost of no-repeat n-gram blocking on the benchmarked workload's inputs (config 2: D = 50, L = 10, R = 20, F = 2048,
V = 10000, T = 20, raw weights of torch.manual_seed(1234), bench.py's seeds 1002..).  Decodes, each with blocking off,
n = 3 and n = 1:

  beam_search_v, beam 5, gt verbs (graph replay), at 100 and at 1000 stacked captions
  greedy (`test`) at 100 captions
  sample_rl(n=5) at 100 captions

All arms of a size run in one process and alternate round by round (the order rotates every round); ms per call by
CUDA events, median [min, max] over `--rounds` rounds.  The card's name, power limit and max SM clock are read in the
same run.

    python tools/ngram_probe.py [--rounds 7] [--out profiles/ngram_probe_b200.json]"""
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
BLOCK = (0, 3, 1)


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
        raise SystemExit("ngram_probe: needs a CUDA device")
    from models import ControllableCaptioningModel
    dev = "cuda:0"
    torch.manual_seed(1234)
    model = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()
    result = {"card": card(), "rounds": args.rounds,
              "workload": "config2 inputs, D=50 L=10 R=20 F=2048 V=10000 T=20, raw weights (torch.manual_seed(1234))"}
    for b, calls in ((100, 5), (1000, 2)):
        det, ds, verbs = (t.to(dev) for t in batch(b))
        arms = {}
        for nb in BLOCK:
            arms[f"beam_search_v_k5_n{nb}"] = (lambda nb=nb: model.beam_search_v((det, ds, verbs), EOS, 5, 1, gt=True,
                                                                                 no_repeat_ngram_size=nb))
            if b == 100:
                arms[f"greedy_n{nb}"] = lambda nb=nb: model.test(det, ds, no_repeat_ngram_size=nb)
                arms[f"sample_rl_x5_n{nb}"] = lambda nb=nb: model.sample_rl(det, ds, seed=1, n=5, no_repeat_ngram_size=nb)

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
        rec = {"calls_per_round": calls}
        for n in names:
            rec[n] = {"ms_per_call": summary(ms[n])}
            print(json.dumps({"captions": b, "arm": n, "ms_per_call": rec[n]["ms_per_call"]["median"],
                              "min": rec[n]["ms_per_call"]["min"], "max": rec[n]["ms_per_call"]["max"]}), flush=True)
        result[str(b)] = rec
        del det, ds, verbs
        torch.cuda.empty_cache()
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
