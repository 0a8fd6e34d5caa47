#!/usr/bin/env python
"""bench.py — captions/sec of the role-shift decoder's beam search on synthetic COCO-Entities-shaped
batches (BASELINE.json metric), on N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE full beam-search decode of one 100-caption batch: the once-per-batch prologue, the 20 decoder
steps (beam 5) and the final back-track, through the reference-facing call
`ControllableCaptioningModel.beam_search_v` of the drop-in `models` package (-> ctypes -> libvsrdec).
Workload = BASELINE config 2 (eval_coco.py --gt shape): 100 captions x beam 5, <=50 detections
x 2048-d, 10 slots x 20 regions, V = 10000, random-init weights (seed 1234).  Multi-GPU = weak scaling:
every rank decodes its own batches, then the finished captions are all-gathered.

What the keys of the JSON line measure (all on the same K timed steps, after W >= 3 warm-up steps):
  value           device-resident throughput: K batches, STACKED `--stack` at a time along the caption axis into one
                  decode call (captions are independent units; a stacked decode is bit-identical to separate ones) on
                  `--lanes` engines/streams; inputs are in HBM before the clock starts; >= 4 distinct batches rotate
  one_at_a_time   the same K batches, one 100-caption decode at a time on one engine and one stream (latency view);
                  p50_* and roofline_b100 refer to it
  e2e             host buffers -> H2D -> beam_search_v -> D2H -> host read through vsrdec.DecodePipeline (same stacking
                  and lanes), every copy inside the timed region
  parity_check    one timed-workload decode verified against the CPU oracle inside this run (see parity_check())

`--dump-outputs DIR` writes what the headline's last timed decode call returned for its last batch (timed step K):
words.npy and gates.npy (ids as float64), log_probs_words.npy and log_probs_gates.npy (float32), each (100, T).
Weights and inputs come from fixed seeds, so two builds run with the same arguments can be compared output for output.

`--impl reference` times the CPU port of the reference's algorithm (oracle/vsr_oracle.py, torch CPU
ops, all host threads) on the SAME workload (100 captions per step); the reference itself is Python and is not
present on the GPU box.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "vsr-guided-cic_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

WORKLOAD = dict(name="coco_entities_eval_gt(config2)", b=100, beam=5, D=50, L=10, R=20, F=2048, V=10000,
                T=20, eos=[3, -1], gt=True)
METRIC = "captions/sec beam-search decode (COCO-Entities shape)"
N_DISTINCT = 4      # distinct synthetic batches per rank that the timed steps rotate over


def workload_config():
    """The `config` object of the JSON line: identical in both arms."""
    w = WORKLOAD
    return {"workload": w["name"], "captions_per_step": w["b"], "beam": w["beam"], "vocab": w["V"],
            "decoder_steps": w["T"], "detections": w["D"], "slots": w["L"], "regions_per_slot": w["R"],
            "weights": "init_weights(seed=1234)", "inputs": f"{N_DISTINCT} distinct batches per rank, rotated",
            "l2": "inputs rotate over 0.8 GB per rank and the weights are 0.29 GB: beyond the 126 MB L2; no flush"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"],
                    bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


def load_ncu_traffic():
    """DRAM bytes per launch of the dominant kernels from the committed ncu run of this build (tools/gpu_ncu_r02.sh ->
    tools/ncu_summary.py -> profiles/r02_ncu_traffic.json); None when the file is missing."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return None


def batch_seed(rank: int, i: int) -> int:
    return 1002 + 16 * rank + i          # rank 0, batch 0 = seed 1002 = the parity tests' config-2 inputs


def make_inputs(rank: int, i: int = 0):
    from tools.synth import synth_inputs
    w = WORKLOAD
    return synth_inputs(w["b"], w["D"], w["L"], w["R"], w["F"], seed=batch_seed(rank, i), vocab_size=w["V"],
                        n_det_range=(10, 50), verb_slots=(2,), verb_vocab_id=17)


def make_inputs_indexed(rank: int, i: int = 0):
    from tools.synth import synth_inputs_indexed
    w = WORKLOAD
    return synth_inputs_indexed(w["b"], w["D"], w["L"], w["R"], w["F"], seed=batch_seed(rank, i),
                                n_det_range=(10, 50), verb_slots=(2,), verb_vocab_id=17)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for ts, r in self.rows if t0 - 0.05 <= ts <= t1 + 0.15 and len(r) >= 8] or \
               [r for _, r in self.rows if len(r) >= 8]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        f = lambda x: float(x) if x.replace(".", "", 1).isdigit() else None
        sm = [f(r[1]) for r in rows if f(r[1]) is not None]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": f(rows[0][2]),
                "power_w_max": max([f(r[3]) or 0.0 for r in rows]), "samples": len(rows), "reasons": reasons}


# ------------------------------------------------------------------------------------------- CPU port
def run_cpu_port(steps, warmup):
    """Times the oracle (CPU restatement of the reference's algorithm) on the full workload: one 100-caption
    beam-search decode per step, rotating over the same batches as the GPU arm.  Returns (captions_per_s, ms_per_step, cores)."""
    from oracle import vsr_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    w = WORKLOAD
    d = O.Dims(seq_len=w["T"], vocab_size=w["V"])
    W = O.init_weights(d, seed=1234)
    batches = [make_inputs(0, i) for i in range(min(N_DISTINCT, warmup + steps))]
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            O.beam_search(W, d, batches[i % len(batches)], w["eos"], w["beam"], 1, use_verbs=True, gt=w["gt"])
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    total = sum(times)
    return w["b"] * len(times) / total, 1e3 * total / len(times), cores


def main_reference(args, rank, world):
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    cps, ms, cores = run_cpu_port(steps, warmup)
    sample = (f"the full workload: {WORKLOAD['b']} captions per step, beam {WORKLOAD['beam']}, {WORKLOAD['T']} decoder "
              f"steps, {steps} timed steps after {warmup} warm-up; oracle/vsr_oracle.py (torch CPU ops, {cores} threads)")
    line = {"impl": "reference", "metric": METRIC, "value": cps, "unit": "captions/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(),
            "cpu_baseline": {"value": cps, "unit": "captions/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": cps, "unit": "captions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- GPU arm
def gemm_flops_per_row_step(dims):
    """Algorithmic FLOPs (2*K*N_out) of the per-step dense contractions this implementation executes:
    SURVEY.md 8d's hoisted formulation (95.54 MFLOP per row-step) minus the xt part of GEMM-A
    (2*E*6H = 12 MFLOP), which is a per-word table lookup here: A = h2->6H + h1->5H,
    B = s_t->(F+A) + h1'->(H+A), D = [att|h2|h1']->4H (+ C = g_t->A in the same launch), E = h2'->V."""
    H, E, F, A, V = dims["H"], dims["E"], dims["F"], dims["A"], dims["V"]
    return {"gemm_a_lstm1_gates": 2 * (H * 6 * H + H * 5 * H),
            "gemm_b_sentinel_h1proj": 2 * (H * (F + A) + H * (H + A)),
            "gemm_d_lstm2_gates": 2 * (F + 2 * H) * 4 * H + 2 * H * A,
            "gemm_e_vocab": 2 * H * V}


def parity_check(model, dev_batch, host_batch, stacked_words, n_check=10):
    """Checks the TIMED workload inside the bench run (rank 0): decodes batch 0 once more, replays the first
    `n_check` captions' device trajectory through the CPU oracle (tests/common.py: verify_device_beam — tie-aware
    top-k check of every decision, accumulated scores, unrolled tokens), and checks that the stacked decode of the
    timed region returned bit-identical captions for that batch.  The oracle is the checker here, never the timed path."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from common import verify_device_beam
    from oracle import vsr_oracle as O
    w = WORKLOAD
    t0 = time.perf_counter()
    eng = model._engine_for(dev_batch)
    (words, gates), (lpw, lpg), _ = eng.beam_search(w["beam"], 1, w["eos"], use_verbs=True, gt=w["gt"])
    hist = [h.cpu()[:, :n_check] for h in eng.history()]
    torch.cuda.synchronize()
    d = O.Dims(seq_len=w["T"], vocab_size=w["V"])
    W = O.init_weights(d, seed=1234)
    statics = tuple(t[:n_check] for t in host_batch)
    v, o_outs, o_lps = verify_device_beam(W, d, statics, w["eos"], w["beam"], hist, True, w["gt"])
    # returned caption = unroll of one of the trajectory's final beams (the best one up to score ties)
    T = w["T"]
    ow = o_outs[0].reshape(n_check, -1, T)
    dw = words[:n_check, 0].cpu()
    unroll_ok = all(any(torch.equal(ow[c, r], dw[c]) for r in range(ow.size(1))) for c in range(n_check))
    best_ok = sum(int(torch.equal(ow[c, 0], dw[c])) for c in range(n_check))
    stacked_same = None if stacked_words is None else bool(torch.equal(stacked_words.cpu().reshape(-1, T), words.cpu().reshape(-1, T)))
    return {"captions_checked": n_check, "decisions": v.decisions, "violations": len(v.violations),
            "in_tie_band": v.in_band, "max_score_err": v.max_score_err, "tokens_are_unroll_of_trajectory": unroll_ok,
            "best_beam_matches_oracle_order": f"{best_ok}/{n_check}",
            "stacked_decode_equals_single_decode": stacked_same,
            "ok": (not v.violations) and unroll_ok and stacked_same is not False,
            "how": "device trajectory of batch 0 replayed through oracle/vsr_oracle.py (forced trajectory), band 2e-3 + 2e-5*|score|",
            "seconds": round(time.perf_counter() - t0, 2)}


def bind_to_gpu_cpus(gpu_index):
    """Pin this rank to its GPU's local CPUs (NVML cpu affinity) BEFORE the pinned host buffers are allocated and first
    touched, so they land on the GPU-local NUMA node (8 ranks pulling 205 MB batches across the inter-socket link is what
    collapsed the round-1 e2e scaling).  Returns a note for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        masks = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = [64 * i + b for i, m in enumerate(masks) for b in range(64) if (m >> b) & 1]
        use = [c for c in cpus if c in os.sched_getaffinity(0)]
        if not use:
            return "no GPU-local cpus in the allowed set"
        os.sched_setaffinity(0, use)
        return f"{len(use)} GPU-local cpus of {os.cpu_count()}"
    except Exception as e:   # noqa: BLE001
        return "unavailable: " + repr(e)[:80]


def dump_outputs(out_dir, outputs):
    """Writes what beam_search_v returned for one batch, (words, gates, lp_words, lp_gates) each (b, T), as
    <out_dir>/<name>.npy: token and gate ids as float64, log-probabilities as float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in zip(("words", "gates", "log_probs_words", "log_probs_gates"), outputs):
        t = t.detach().cpu()
        t = t.float() if t.is_floating_point() else t.double()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


def main_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    from models import ControllableCaptioningModel
    from vsrdec import DecodePipeline
    w = WORKLOAD
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    gpu_index = (local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                 int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
    bind_note = bind_to_gpu_cpus(gpu_index) if not args.no_bind else "off"
    if world > 1:
        # stdout carries exactly one JSON line: NCCL logs (its version banner at NCCL_DEBUG=VERSION/WARN) go to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    S, n_lanes, K = max(1, args.stack), max(1, args.lanes), args.steps
    b, T = w["b"], w["T"]

    torch.manual_seed(1234)                       # the eval scripts' seed (eval_coco.py:22)
    model = ControllableCaptioningModel(T, w["V"], 2, verb_tables=({}, {})).to(dev).eval()
    lane_models = [model]
    for _ in range(n_lanes - 1):
        replica = ControllableCaptioningModel(T, w["V"], 2, verb_tables=({}, {})).to(dev).eval()
        replica.load_state_dict(model.state_dict())
        lane_models.append(replica)
    host = [tuple(t.pin_memory() for t in make_inputs(rank, i)) for i in range(N_DISTINCT)]
    dev_single = [tuple(t.to(dev) for t in hb) for hb in host]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host[0])
    # stacked device-resident inputs: set j holds batches (j, j+1, .., j+S-1) mod N_DISTINCT along the caption axis
    n_sets = max(2 * n_lanes, 2)
    dev_stacked = [tuple(torch.cat([dev_single[(j + i) % N_DISTINCT][x] for i in range(S)], 0) for x in range(3))
                   for j in range(n_sets)] if S > 1 else dev_single

    def gather(words):
        if world == 1:
            return words
        bufs = [torch.empty_like(words) for _ in range(world)]
        dist.all_gather(bufs, words)
        return torch.cat(bufs, 0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(x):
        if world > 1:
            tt = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            return float(tt)
        return x

    # ---- one decode at a time (latency view): K batches of 100 captions, one engine, one stream
    def decode_single(i):
        (words, gates), (lpw, lpg) = model.beam_search_v(dev_single[i % N_DISTINCT], w["eos"], w["beam"], 1, gt=w["gt"])
        return gather(words)

    def timed_single(steps):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        barrier()
        ev[0].record()
        for i in range(steps):
            decode_single(i)
            ev[i + 1].record()
        barrier()
        return max_over_ranks(ev[0].elapsed_time(ev[-1])), [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]

    for i in range(max(args.warmup, 3 * N_DISTINCT)):      # per input buffer: eager, graph capture, replay
        decode_single(i)
    eng = model._eng
    sampler = ClockSampler(gpu_index)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    t_wall0 = time.time()
    l0 = eng.launch_count()
    single_ms, per_ms = timed_single(K)
    single_launches = eng.launch_count() - l0

    # ---- headline: the same K batches, stacked S at a time into one decode call, `n_lanes` calls in flight
    lanes = [torch.cuda.Stream(dev) for _ in range(n_lanes)]
    groups = [min(S, K - g0) for g0 in range(0, K, S)]      # batches per decode call
    last = {}

    def stacked_run():
        cur = torch.cuda.current_stream(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(cur)
        for ln in lanes:
            ln.wait_event(e0)
        for gi, n in enumerate(groups):
            ln = gi % n_lanes
            with torch.cuda.stream(lanes[ln]):
                # lane ln rotates over its own stacked sets: ln, ln + n_lanes, ...
                sset = dev_stacked[(ln + n_lanes * (gi // n_lanes)) % len(dev_stacked)]
                statics = tuple(t[:n * b] for t in sset)
                (words, gates), (lpw, lpg) = lane_models[ln].beam_search_v(statics, w["eos"], w["beam"], 1, gt=w["gt"])
                last["words"], last["set"], last["n"] = gather(words), (ln + n_lanes * (gi // n_lanes)) % len(dev_stacked), n
                last["outputs"] = (words, gates, lpw, lpg)
        for ln in lanes:
            ev = torch.cuda.Event()
            ev.record(ln)
            cur.wait_event(ev)
        e1.record(cur)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))
    for _ in range(3):                                      # every (lane, set, group size): eager, capture, replay
        stacked_run()
    l2 = sum(m._eng.launch_count() for m in lane_models)
    stacked_ms = stacked_run()
    stacked_launches = sum(m._eng.launch_count() for m in lane_models) - l2
    clocks = sampler.stop(t_wall0, time.time()) if rank == 0 else None
    value = world * b * K / (stacked_ms * 1e-3)

    # ---- end to end: pinned host batches -> H2D -> beam_search_v -> D2H -> host, through the package's pipeline
    result = {}

    def e2e_measure(host_batches, indexed, stack):
        pipe = DecodePipeline(lane_models, w["eos"], w["beam"], 1, gt=w["gt"], indexed=indexed, buffers=2 * n_lanes,
                              stack=stack, post=gather)

        def e2e_run(steps):
            for words, gates, lpw, lpg in pipe.run(host_batches[i % len(host_batches)] for i in range(steps)):
                result["words"], result["gates"], result["lps"] = words, gates, (lpw, lpg)
        for _ in range(3):                                  # every (lane, buffer, group size): eager, capture, replay
            e2e_run(K)
        barrier()
        t_e0 = time.perf_counter()
        e2e_run(K)
        barrier()
        return max_over_ranks(time.perf_counter() - t_e0)

    # (the materialised input format is H2D-bound: smaller groups pipeline the copies better over K = 20 steps)
    S_e2e = max(1, args.e2e_stack)
    e2e_s = e2e_measure(host, False, S_e2e)
    e2e_value = world * b * K / e2e_s
    d2h_bytes = int(sum(t.numel() * t.element_size() for t in (result["words"], result["gates"]) + result["lps"]))

    # ---- the same e2e loop through the index-form entry point (SURVEY 8 f3, vsr_prologue_indexed): the slots
    # arrive as int32 indices into the detections instead of materialised (b,L,R,F) tiles
    host_i = [tuple(t.pin_memory() for t in make_inputs_indexed(rank, i)) for i in range(N_DISTINCT)]
    S_idx = max(1, args.idx_stack)
    e2e_idx_s = e2e_measure(host_i, True, S_idx)
    h2d_idx_bytes = sum(t.numel() * t.element_size() for t in host_i[0])
    del host_i

    # ---- secondary workload (SURVEY 8d config 5): teacher-forced forward, B=100, T=20, D=100 (train.py:99-103 shape)
    fwd = None
    if rank == 0:
        gq = torch.Generator().manual_seed(1005)
        f_det = torch.relu(torch.randn((100, 100, w["F"]), generator=gq)).to(dev)
        f_caps = torch.randint(0, w["V"], (100, T), generator=gq).to(dev)
        f_ctrl = torch.relu(torch.randn((100, T, w["R"], w["F"]), generator=gq))
        f_nv = torch.randint(1, w["R"] + 1, (100, T), generator=gq)
        f_ctrl = (f_ctrl * (torch.arange(w["R"])[None, None, :] < f_nv[:, :, None]).unsqueeze(-1)).to(dev)
        for _ in range(3):
            model((f_det,), (f_caps, f_ctrl))
        torch.cuda.synchronize(dev)
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_fwd = 5
        fe0.record()
        for _ in range(n_fwd):
            model((f_det,), (f_caps, f_ctrl))
        fe1.record()
        torch.cuda.synchronize(dev)
        f_ms = fe0.elapsed_time(fe1) / n_fwd
        fwd = {"workload": "xe_forward(config5): B=100, T=20, D=100, full (B,T,V) log-prob output", "ms_per_forward": f_ms,
               "row_steps_per_s": 100 * T / (f_ms * 1e-3), "n_gpus": 1}
        del f_det, f_caps, f_ctrl
    # ---- eval pre-step (SURVEY 8 f2): role ordering of 100 synthetic captions (S-level sorter + R-level network + host
    # bookkeeping, vsrdec.preorder.RoleOrderer), wall clock around the call incl. its two device calls and host reads
    prestep = None
    if rank == 0:
        from models import S_SSP, SinkhornNet
        from tools.synth import synth_eval_captions
        from vsrdec.preorder import RoleOrderer
        sort_net, sk_net = S_SSP().to(dev).eval(), SinkhornNet(10, 20, 0.1).to(dev).eval()
        orderer = RoleOrderer(sort_net, sk_net, sinkhorn_len=10, fixed_len=10)
        caps = synth_eval_captions(C=100, seed=5)
        sp = caps["seqs_perm"].to(dev)
        a_ = (caps["control_verb"], caps["det_seqs_v"], caps["det_seqs_sr"], caps["verb_list"], sp, caps["slot_valid"])
        for _ in range(2):
            orderer.order(*a_)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        n_pre = 5
        for _ in range(n_pre):
            orderer.order(*a_)
        torch.cuda.synchronize(dev)
        pre_ms = (time.perf_counter() - t0) * 1e3 / n_pre
        n_s = int(sum((cv != 0).sum() for cv in caps["control_verb"]))
        prestep = {"workload": "role ordering of 100 synthetic captions (1-3 verbs, 3-8 slots each; eval_coco.py:127-237)",
                   "ms_per_100_captions": pre_ms, "s_level_problems": n_s,
                   "how": "wall clock around vsrdec.preorder.RoleOrderer.order: host bookkeeping + one S_SSP.generate_batch + one "
                          "SinkhornNet.assign + host reads of their results"}
        sort_net.close(); sk_net.close()
        del sort_net, sk_net, orderer, sp
    barrier()

    # ---- per-kernel times: profiled (eager, CUDA events around every phase and every step) repeats of a decode, once
    # for the stacked call of the headline and once for the single 100-caption call
    def profile(statics, n_prof):
        acc, total, steps_ms = {}, 0.0, []
        eng.set_profiling(True)
        for _ in range(n_prof):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            model.beam_search_v(statics, w["eos"], w["beam"], 1, gt=w["gt"])
            e1.record()
            torch.cuda.synchronize(dev)
            total += e0.elapsed_time(e1)
            for name, ms, calls in eng.phase_times():
                a = acc.setdefault(name, [0.0, 0])
                a[0] += ms
                a[1] += calls
            steps_ms += eng.step_times()
        eng.set_profiling(False)
        return {n: (v[0] / n_prof, v[1] / n_prof) for n, v in acc.items()}, total / n_prof, steps_ms

    line = None
    if rank == 0:
        n_prof = min(K, 5)
        ph1, prof1_ms, step1_ms = profile(dev_single[0], n_prof)
        parent, word, gate, score = [x.cpu() for x in eng.history()]
        phS, profS_ms, _ = profile(dev_stacked[0], n_prof) if S > 1 else (ph1, prof1_ms, None)
        dims = dict(H=1000, E=1000, F=w["F"], A=512, V=w["V"])
        k = w["beam"]
        fl = gemm_flops_per_row_step(dims)
        gemm_names = list(fl.keys())
        traffic = load_ncu_traffic() or {}

        def gemm_roofline(ph, prof_ms, caps, what):
            rows_total = caps * 1 + caps * k * (T - 1)                  # row-steps per decode call
            gemm_ms = sum(ph[n][0] for n in gemm_names)
            gemm_flops = sum(fl.values()) * rows_total
            achieved_tf = gemm_flops / (gemm_ms * 1e-3) / 1e12
            peak_tf = peaks["bf16_tflops_sustained"]
            f8 = "f8" in eng.gemm_kind()
            return {"kernel": ("k_gemm_tc / k_gemm_tcp, the four per-step GEMM phases: tcgen05.mma kind::f16 (x_hi*w_hi) + 2x kind::f8f6f4 e4m3 "
                               "(x_hi*w_lo, x_lo*w_hi) into one fp32 TMEM accumulator, TMA-fed" if f8 else
                               "k_gemm_tc / k_gemm_tcp, the four per-step GEMM phases: 3x tcgen05.mma kind::f16 (f16x3 hi/lo split), TMA + TMEM"),
                    "gemm_kind": eng.gemm_kind(),
                    "describes": what, "bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                    "frac": achieved_tf / peak_tf,
                    "traffic": traffic.get("gemm_bytes_per_launch_b%d" % caps, traffic.get("gemm_bytes_per_launch_b1000" if caps > 100 else "gemm_bytes_per_launch_b100")),
                    "traffic_source": traffic.get("source"),
                    "peak_source": f"{peaks['source']} bf16_tflops_sustained (MEASURED_PEAKS.json)",
                    "passes": 3, "f16_equivalent_passes": 2 if f8 else 3,
                    "issued_tflops": achieved_tf * (2 if f8 else 3), "issued_frac": achieved_tf * (2 if f8 else 3) / peak_tf,
                    "issued_note": "tensor-pipe time in units of one fp16 pass (an e4m3 pass runs at twice the fp16 rate)",
                    "flops_per_decode": gemm_flops, "ms_per_decode": gemm_ms,
                    "launches_per_decode": sum(ph[n][1] for n in gemm_names), "share_of_step": gemm_ms / prof_ms,
                    "timing": f"CUDA events around every GEMM launch of {n_prof} profiled (eager) decodes of the timed workload"}
        roofline = gemm_roofline(phS, profS_ms, S * b, f"the headline's decode call: {S} stacked batches = {S * b} captions, one call on one stream")
        roofline_b100 = gemm_roofline(ph1, prof1_ms, b, "one 100-caption decode (one_at_a_time)")
        # attention kernel against the HBM roofline: exact algorithmic bytes from the decode's slot-pointer trajectory
        ds = host[0][1]
        ptr = torch.zeros((b, 1), dtype=torch.long)
        nvalid = (ds.sum(-1) != 0).sum(-1)                       # (b, L) valid regions per slot
        att_bytes, uniq_bytes = 0, 0
        for t in range(T):
            cur = ptr.size(1)
            nv = torch.gather(nvalid, 1, ptr)                    # (b, cur)
            per_row = (dims["F"] + 3 * dims["A"] + dims["H"]) * 4 + (dims["F"] + 2) * 4
            att_bytes += int((nv * (dims["F"] + dims["A"]) * 4).sum()) + b * cur * per_row
            for c in range(b):                                   # a slot tile shared by several beams counted once
                uniq_bytes += sum(int(nvalid[c, s]) for s in set(ptr[c].tolist())) * (dims["F"] + dims["A"]) * 4
            uniq_bytes += b * cur * per_row
            ptr = torch.clamp(torch.gather(ptr, 1, parent[t].long()) + gate[t].long(), 0, w["L"] - 1)
        att_ms = ph1["attend_gate"][0]
        att_gbs = att_bytes / (att_ms * 1e-3) / 1e9
        roofline_att = {"kernel": "k_attend (slot attention + shift gate, one CTA per beam row)", "bound": "hbm",
                        "describes": "one 100-caption decode (one_at_a_time)", "achieved": att_gbs,
                        "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": att_gbs / peaks["hbm_gbs"],
                        "traffic": traffic.get("attend_bytes_per_launch_b100"), "traffic_source": traffic.get("source"),
                        "bytes_per_decode": att_bytes, "unique_bytes_per_decode": uniq_bytes, "ms_per_decode": att_ms,
                        "note": "achieved counts SURVEY 8d's algorithmic bytes (every beam row reads its slot tile); the beams of a "
                                "caption mostly share a tile, so L2 serves the repeats and DRAM sees about unique_bytes_per_decode"}
        roofline_att_stacked = None
        if S > 1:
            attS_ms = phS["attend_gate"][0]
            attS_gbs = S * att_bytes / (attS_ms * 1e-3) / 1e9
            roofline_att_stacked = {"kernel": roofline_att["kernel"], "bound": "hbm",
                                    "describes": f"the headline's decode call ({S * b} captions)", "achieved": attS_gbs,
                                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": attS_gbs / peaks["hbm_gbs"],
                                    "traffic": traffic.get("attend_bytes_per_launch_b1000"), "traffic_source": traffic.get("source"),
                                    "bytes_per_decode": S * att_bytes, "ms_per_decode": attS_ms,
                                    "note": f"algorithmic bytes estimated as {S} x those of batch 0's trajectory (the stacked batches are "
                                            "drawn from the same distribution); L2 serves the beams that share a slot tile, so the "
                                            "algorithmic rate can exceed the DRAM rate (traffic / launch time)"}
        check = parity_check(model, dev_single[0], host[0], None)
        # the stacked decode of set 0 holds batch 0 in its first 100 rows: must equal the single decode bit for bit
        (w_st, _), _ = model.beam_search_v(dev_stacked[0], w["eos"], w["beam"], 1, gt=w["gt"])
        (w_si, _), _ = model.beam_search_v(dev_single[0], w["eos"], w["beam"], 1, gt=w["gt"])
        torch.cuda.synchronize(dev)
        check["stacked_decode_equals_single_decode"] = bool(torch.equal(w_st[:b], w_si))
        check["ok"] = check["ok"] and check["stacked_decode_equals_single_decode"]
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_cps, cpu_ms, cores = run_cpu_port(1, 1)
            cpu = {"value": cpu_cps, "unit": "captions/s", "cores": cores, "kind": "port",
                   "sample": f"the full workload: one {b}-caption decode timed after one warm-up decode of "
                             f"oracle/vsr_oracle.py (torch CPU ops, {cores} threads)"}
        line = {"metric": METRIC, "value": value, "unit": "captions/s", "n_gpus": world, "steps": K,
                "warmup": args.warmup, "ms_per_step": stacked_ms / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(),
                "execution": {"stack": S, "lanes": n_lanes, "decode_calls": len(groups),
                              "parallelism": f"caption-sharded x{world} (weights replicated, one all_gather of captions per batch)",
                              "note": f"value: the K batches are decoded {S} at a time (stacked along the caption axis into one "
                                      f"beam_search_v call) on {n_lanes} engine(s)/stream(s); one_at_a_time: one batch per call"},
                "gpu_launches": int(stacked_launches) * world,
                "one_at_a_time": {"value": world * b * K / (single_ms * 1e-3), "unit": "captions/s", "ms_per_step": single_ms / K,
                                  "gpu_launches": int(single_launches) * world, "p50_decode_ms": statistics.median(per_ms)},
                "p50_step_latency_ms": statistics.median(step1_ms) if step1_ms else None,
                "p95_step_latency_ms": (sorted(step1_ms)[int(0.95 * (len(step1_ms) - 1))] if step1_ms else None),
                "step_latency_note": f"CUDA events around each of the {T} decoder steps (decoder step + beam selection/reorder) of "
                                     f"{n_prof} eager 100-caption decodes; inside the CUDA-graph replay a step takes p50_decode_ms / {T}",
                "e2e": {"value": e2e_value, "unit": "captions/s", "h2d_bytes_per_step": h2d_bytes,
                        "d2h_bytes_per_step": d2h_bytes, "ms_per_step": 1e3 * e2e_s / K,
                        "h2d_gbs": world * h2d_bytes * K / e2e_s / 1e9, "cpu_binding": bind_note,
                        "pipeline": f"vsrdec.DecodePipeline: stack {S_e2e}, {n_lanes} lanes, {2 * n_lanes} input buffers; H2D (copy stream), "
                                    "decodes and D2H + host read of finished results overlap; all inside the timed region"},
                "e2e_indexed": {"value": world * b * K / e2e_idx_s, "unit": "captions/s",
                                "h2d_bytes_per_step": h2d_idx_bytes, "d2h_bytes_per_step": d2h_bytes,
                                "ms_per_step": 1e3 * e2e_idx_s / K, "stack": S_idx,
                                "entry": "beam_search_v_indexed / vsr_prologue_indexed: slots as int32 indices into the detections"},
                "parity_check": check,
                "forward_teacher": fwd,
                "eval_prestep": prestep,
                "roofline": roofline, "roofline_b100": roofline_b100, "roofline_attend": roofline_att, "roofline_attend_stacked": roofline_att_stacked,
                "phases_ms_per_decode": {n: v[0] for n, v in ph1.items()},
                "phases_ms_per_stacked_decode": {n: v[0] for n, v in phS.items()} if S > 1 else None,
                "profiled_ms_per_decode": prof1_ms,
                "clocks": clocks}
        if cpu is not None:
            line["cpu_baseline"] = cpu
    # ---- N > 1: the all-gathered captions of the last stacked decode, checked on rank 0 against its own re-decode of
    # another rank's inputs (captions are independent units, so any GPU must produce the same tokens)
    if world > 1:
        gathered = last["words"]                                 # (world * n * b, T): rank-major blocks
        if rank == 0:
            n, sset = last["n"], last["set"]
            ok, checked = True, []
            for r in range(1, min(world, 3)):
                # rank r's stacked set `sset` = its batches (sset + i) % N_DISTINCT, i < n
                st = tuple(torch.cat([t for t in xs], 0).to(dev) for xs in
                           zip(*[make_inputs(r, (sset + i) % N_DISTINCT) for i in range(n)]))
                (w_r, _), _ = model.beam_search_v(st, w["eos"], w["beam"], 1, gt=w["gt"])
                torch.cuda.synchronize(dev)
                same = bool(torch.equal(w_r, gathered[r * n * b:(r + 1) * n * b]))
                ok = ok and same
                checked.append(r)
            line["parity_check"]["gathered_blocks_equal_rank0_redecode"] = {"ranks": checked, "equal": ok}
            line["parity_check"]["ok"] = line["parity_check"]["ok"] and ok
        dist.barrier()
    if rank == 0:
        if args.dump_outputs:
            # the last timed step is the last 100-caption batch of the last timed decode call
            dump_outputs(args.dump_outputs, [t[-b:] for t in last["outputs"]])
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bind", action="store_true", help="do not pin the rank to its GPU's local CPUs")
    ap.add_argument("--stack", type=int, default=10, help="batches stacked along the caption axis per decode call")
    ap.add_argument("--idx-stack", type=int, default=5, help="batches per decode call of the index-form e2e loop")
    ap.add_argument("--e2e-stack", type=int, default=1, help="batches per decode call of the e2e loop (materialised inputs)")
    ap.add_argument("--lanes", type=int, default=2, help="decode calls in flight per GPU (engines on their own streams)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the run, write the outputs of the last timed step "
                    "(the words, gates and log-probs the headline's decode call returned for its last batch) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        main_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the decoder path has no CPU fallback "
                         "(use --impl reference for the CPU port)")
    if world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    main_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
