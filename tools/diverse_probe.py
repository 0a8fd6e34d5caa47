"""Cost of diverse beam search on the benchmarked workload's inputs (config 2: D = 50, L = 10, R = 20, F = 2048,
V = 10000, T = 20, raw weights of torch.manual_seed(1234), bench.py's seeds 1002..).  beam_search_v with gt verbs
(graph replay), at 100 and at 1000 stacked captions per call:

  beam 6: one group (plain), 2 groups and 3 groups
  beam 5: one group (plain) and 5 groups

with diversity_penalty = 1.0.  All arms of a size run in one process and alternate round by round (the order rotates
every round); ms per call by CUDA events, median [min, max] over `--rounds` rounds.  Per arm it also reports the share
of distinct captions among the beam_size captions returned per input (out_size = beam_size); on random-init weights
that is a sanity number, not a quality claim.  The card's name, power limit and max SM clock are read in the same run.

    python tools/diverse_probe.py [--rounds 7] [--out profiles/diverse_probe_b200.json]"""
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
PENALTY = 1.0
SETTINGS = ((6, 1), (6, 2), (6, 3), (5, 1), (5, 5))     # (beam, groups)


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


def distinct_share(words):
    """Distinct captions among the beam captions of every input, summed over inputs, over all captions returned."""
    b, k, _ = words.shape
    w = words.cpu().tolist()
    return sum(len({tuple(y) for y in w[c]}) for c in range(b)) / (b * k)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diverse_probe: needs a CUDA device")
    from models import ControllableCaptioningModel
    dev = "cuda:0"
    torch.manual_seed(1234)
    model = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()
    result = {"card": card(), "rounds": args.rounds, "diversity_penalty": PENALTY,
              "workload": "config2 inputs, D=50 L=10 R=20 F=2048 V=10000 T=20, raw weights (torch.manual_seed(1234))"}
    for b, calls in ((100, 5), (1000, 2)):
        det, ds, verbs = (t.to(dev) for t in batch(b))

        def decode(k, g, out_size=1):
            return model.beam_search_v((det, ds, verbs), EOS, k, out_size, gt=True, num_beam_groups=g,
                                       diversity_penalty=PENALTY if g > 1 else 0.0)

        arms = {f"beam{k}_groups{g}": (lambda k=k, g=g: decode(k, g)) for k, g in SETTINGS}

        def run(fn, n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        for fn in arms.values():                          # warm: every shape, eager + graph capture + replay
            run(fn, 3)
        names = list(arms)
        ms = {n: [] for n in names}
        for r in range(args.rounds):
            rot = names[r % len(names):] + names[:r % len(names)]
            for n in rot:
                ms[n].append(run(arms[n], calls))
        rec = {"calls_per_round": calls}
        for (k, g), n in zip(SETTINGS, names):
            (words, _), _ = decode(k, g, out_size=k)
            rec[n] = {"ms_per_call": summary(ms[n]), "distinct_caption_share": distinct_share(words)}
            print(json.dumps({"captions": b, "arm": n, "ms_per_call": rec[n]["ms_per_call"]["median"],
                              "min": rec[n]["ms_per_call"]["min"], "max": rec[n]["ms_per_call"]["max"],
                              "distinct_caption_share": rec[n]["distinct_caption_share"]}), flush=True)
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
