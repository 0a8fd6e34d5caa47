"""Half-precision region features (fp16 / bf16) against fp32 on the benchmarked workload (config 2: beam 5, D = 50,
L = 10, R = 20, F = 2048, V = 10000, raw weights of torch.manual_seed(1234), bench.py's seeds 1002..1005).

The inputs are generated once in fp32 and converted to each dtype before anything is timed, as a dataset stored in
that dtype would be.  All arms run in one process and alternate round by round (the order rotates every round); the
report is the median [min, max] over `--rounds` rounds.

  1. End to end: pinned host batches through vsrdec.DecodePipeline with two lanes, as bench.py's e2e does: the
     materialised form (det + det_seqs, one batch per decode call) and the index form (det + slot_index, five batches
     per call).  Captions/s and GB/s of host-to-device input copies.
  2. Device resident: ms per 100-caption call and per 1000-caption stacked call (CUDA events, graph replay), and, in
     separate rounds with the phase profiler on, the prologue and attention phase times of one call.
  3. For every size timed, whether the half-precision arm's outputs (words, gates, both log-probs) equal bit for bit
     those of a decode of its fp32 upcast.

    python tools/half_probe.py [--rounds 7] [--batches 40] [--out profiles/half_probe_b200.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "vsr-guided-cic_b200")):
    sys.path.insert(0, p)
import torch  # noqa: E402

from tools.synth import synth_inputs, synth_inputs_indexed  # noqa: E402

DTYPES = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}
N_DISTINCT = 4
EOS = [3, -1]


def batch(seed, b=100):
    return synth_inputs(b, 50, 10, 20, 2048, seed=seed, vocab_size=10000, n_det_range=(10, 50), verb_slots=(2,),
                        verb_vocab_id=17)


def batch_indexed(seed, b=100):
    return synth_inputs_indexed(b, 50, 10, 20, 2048, seed=seed, n_det_range=(10, 50), verb_slots=(2,),
                                verb_vocab_id=17)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def in_dtype(statics, dt):
    """features (the floating-point tensors except the float64 verbs) in dt; slot_index and verbs unchanged"""
    return tuple(t.to(dt) if t.dtype == torch.float32 else t for t in statics)


def upcast(statics):
    return tuple(t.float() if t.dtype in (torch.float16, torch.bfloat16) else t for t in statics)


def nbytes(statics):
    return sum(t.numel() * t.element_size() for t in statics)


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "all": xs}


def same_outputs(a, b):
    return all(torch.equal(x.cpu(), y.cpu()) for x, y in zip(a, b))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--batches", type=int, default=40, help="100-caption batches per timed end-to-end run")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("half_probe: needs a CUDA device")
    from models import ControllableCaptioningModel
    from vsrdec import DecodePipeline
    dev = "cuda:0"
    torch.manual_seed(1234)
    model = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()

    def replica():
        r = ControllableCaptioningModel(20, 10000, 2, verb_tables=({}, {})).to(dev).eval()
        r.load_state_dict(model.state_dict())
        return r

    # one pair of lane engines per arm: an engine keeps 16 decode graphs, fewer than three arms' buffers need
    lanes = {n: [replica(), replica()] for n in DTYPES}
    result = {"card": card(), "rounds": args.rounds,
              "workload": "config2 beam 5, D=50 L=10 R=20 F=2048 V=10000, raw weights (torch.manual_seed(1234))"}

    def beam(m, statics, indexed=False):
        fn = m.beam_search_v_indexed if indexed else m.beam_search_v
        (w, g), (lw, lg) = fn(statics, EOS, 5, 1, gt=True)
        return w, g, lw, lg

    # ---------------------------------------------------------------- 1. end to end
    mat = [batch(1002 + i) for i in range(N_DISTINCT)]
    idx = [batch_indexed(1002 + i) for i in range(N_DISTINCT)]
    e2e = {}
    for form, base, indexed, stack in (("materialised", mat, False, 1), ("indexed", idx, True, 5)):
        host = {n: [tuple(t.pin_memory() for t in in_dtype(hb, dt)) for hb in base] for n, dt in DTYPES.items()}
        pipes = {n: DecodePipeline(lanes[n], EOS, 5, 1, gt=True, indexed=indexed, buffers=4, stack=stack) for n in DTYPES}
        K = args.batches

        def run(n):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            outs = list(pipes[n].run(host[n][i % N_DISTINCT] for i in range(K)))
            torch.cuda.synchronize()
            return time.perf_counter() - t0, outs

        for n in DTYPES:                                   # every (lane, buffer, group size): eager, capture, replay
            for _ in range(3):
                run(n)
        secs = {n: [] for n in DTYPES}
        order = list(DTYPES)
        for r in range(args.rounds):
            for n in order[r % 3:] + order[:r % 3]:
                secs[n].append(run(n)[0])
        rec = {"stack": stack, "lanes": 2, "batches_per_run": K, "captions_per_batch": 100}
        for n in DTYPES:
            bpb = nbytes(host[n][0])
            cps = [K * 100 / s for s in secs[n]]
            gbs = [K * bpb / s / 1e9 for s in secs[n]]
            rec[n] = {"h2d_bytes_per_batch": bpb, "captions_per_s": summary(cps), "h2d_GB_per_s": summary(gbs)}
            if n != "fp32":        # pipeline outputs of the half arm against direct decodes of the upcast batches
                _, outs = run(n)
                ok = True
                for i in range(N_DISTINCT):
                    want = beam(model, tuple(t.to(dev) for t in upcast(host[n][i])), indexed)
                    ok = ok and same_outputs(outs[i], want)
                rec[n]["outputs_equal_upcast"] = ok
            print(json.dumps({"e2e": form, "dtype": n, "captions_per_s": rec[n]["captions_per_s"]["median"],
                              "h2d_GB_per_s": rec[n]["h2d_GB_per_s"]["median"],
                              "outputs_equal_upcast": rec[n].get("outputs_equal_upcast")}), flush=True)
        e2e[form] = rec
        del host, pipes
    result["e2e"] = e2e

    # ---------------------------------------------------------------- 2. device resident
    sizes = {100: (mat[0], 20), 1000: (tuple(torch.cat(x, 0) for x in zip(*[batch(1002 + i) for i in range(10)])), 5)}
    dres = {}
    for b, (host, calls) in sizes.items():
        dstat = {n: tuple(t.to(dev) for t in in_dtype(host, dt)) for n, dt in DTYPES.items()}

        def run(n, k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(k):
                res = beam(model, dstat[n])
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k, res

        rec = {"calls_per_round": calls, "input_bytes": {n: nbytes(dstat[n]) for n in DTYPES}}
        for n in DTYPES:
            _, got = run(n, 3)                             # warm: eager, graph capture, replay
            if n != "fp32":
                up = upcast(dstat[n])
                rec[f"{n}_outputs_equal_upcast"] = same_outputs(got, beam(model, up))
                del up
        ms = {n: [] for n in DTYPES}
        order = list(DTYPES)
        for r in range(args.rounds):
            for n in order[r % 3:] + order[:r % 3]:
                ms[n].append(run(n, calls)[0])
        # phase profiler (no graph replay; separate rounds)
        model._eng.set_profiling(True)
        phases = {n: {"prologue": [], "attend_gate": []} for n in DTYPES}
        for r in range(args.rounds):
            for n in order[r % 3:] + order[:r % 3]:
                beam(model, dstat[n])
                torch.cuda.synchronize()
                pt = {name: t for name, t, _ in model._eng.phase_times()}
                for k in phases[n]:
                    phases[n][k].append(pt[k])
        model._eng.set_profiling(False)
        for n in DTYPES:
            rec[n] = {"ms_per_call": summary(ms[n]),
                      "profiled_phase_ms": {k: summary(v) for k, v in phases[n].items()}}
            print(json.dumps({"captions": b, "dtype": n, "ms_per_call": rec[n]["ms_per_call"]["median"],
                              **{f"{k}_ms": rec[n]["profiled_phase_ms"][k]["median"] for k in phases[n]},
                              "outputs_equal_upcast": rec.get(f"{n}_outputs_equal_upcast")}), flush=True)
        dres[str(b)] = rec
        del dstat
    result["device_resident"] = dres
    print(json.dumps(result["card"]))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
