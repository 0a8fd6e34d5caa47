"""Cost of attention capture: beam_search_v(..., return_attention=True) against the plain call on the benchmarked
workload (config 2: beam 5, D = 50, L = 10, R = 20, V = 10000, raw init_weights(seed 1234)), at 100 captions (one
batch) and 1000 captions (ten batches stacked along the caption axis into one call).

Both arms run in the same process and alternate round by round; each round times `--calls` back-to-back calls of one
arm with CUDA events (graph replay, warmed), and the report is the median over `--rounds` rounds.  The captured arm's
time includes turning capture on and off and the gather of the returned attention (vsr_get_attention).

    python tools/attention_probe.py [--rounds 7] [--out profiles/attention_probe_b200.json]"""
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


def batch(seed, b=100):
    return synth_inputs(b, 50, 10, 20, 2048, seed=seed, vocab_size=10000, n_det_range=(10, 50), verb_slots=(2,),
                        verb_vocab_id=17)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_probe: needs a CUDA device")
    from models import ControllableCaptioningModel
    dev = "cuda:0"
    torch.manual_seed(1234)
    m = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()
    sets = {100: (batch(1002), 20), 1000: (tuple(torch.cat(x, 0) for x in zip(*[batch(1002 + i) for i in range(10)])), 5)}
    result = {"card": card(), "workload": "config2 beam 5, D=50 L=10 R=20 F=2048 V=10000, raw weights seed 1234",
              "rounds": args.rounds, "sizes": {}}
    for b, (host, calls) in sets.items():
        statics = tuple(x.to(dev) for x in host)

        def run(att, n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                res = m.beam_search_v(statics, [3, -1], 5, 1, gt=True, return_attention=att)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n, res

        _, ref = run(False, 3)          # warm: eager, graph capture, replay of both arms
        _, got = run(True, 3)
        same = all(torch.equal(x, y) for x, y in zip(ref[0] + ref[1], got[0] + got[1]))
        off, on = [], []
        for r in range(args.rounds):
            arms = (False, True) if r % 2 == 0 else (True, False)
            for att in arms:
                (on if att else off).append(run(att, calls)[0])
        ratio = [b_ / a_ for a_, b_ in zip(off, on)]
        result["sizes"][str(b)] = {
            "calls_per_round": calls, "ms_off": off, "ms_on": on,
            "median_ms_off": statistics.median(off), "median_ms_on": statistics.median(on),
            "median_overhead_pct": 100.0 * (statistics.median(ratio) - 1.0),
            "outputs_identical": same}
        print(json.dumps({"captions": b, **{k: v for k, v in result["sizes"][str(b)].items() if k.startswith("median")},
                          "outputs_identical": same}), flush=True)
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
