"""Golden vectors of the R-level SSP step from the UNMODIFIED reference (build container only).

    python tests/golden/make_golden_ssp.py     ->  tests/golden/ssp_small.pt

Imports /root/reference/models/sinkhorn_network.py (SinkhornNet) and /root/reference/utils/tools.py (verb_rank_merge),
runs them on seeded inputs and stores inputs + outputs: the pin for oracle/ssp_oracle.py."""
import importlib.util
import os
import random
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("VSR_REFERENCE_ROOT", "/root/reference")


def load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    sk = load(os.path.join(REF, "models", "sinkhorn_network.py"), "_ref_sinkhorn_network")
    tools = load(os.path.join(REF, "utils", "tools.py"), "_ref_tools")
    torch.manual_seed(1234)
    net = sk.SinkhornNet(10, 20, 0.1).eval()
    from oracle import ssp_oracle as S
    seq = S.synth_seq(6, 10, 77)
    with torch.no_grad():
        out = net(seq)
    rnd = random.Random(5)
    merges = []
    for _ in range(200):
        n = rnd.randint(2, 8)
        pool = list(range(10))
        la = rnd.sample(pool, rnd.randint(1, n))
        lb = rnd.sample(pool, rnd.randint(1, n))
        merges.append((list(la), list(lb), tools.verb_rank_merge(list(la), list(lb))))
    # the oracle's matrix for a second input, computed where these vectors are made: a test host that reproduces it
    # bit for bit rounds float32 like this one (tests/test_oracle_ssp.py then demands the reference's matrix bit for bit)
    with torch.no_grad():
        probe = {"seed_x": 78, "matrix": S.forward(S.init_weights(10, 1234), S.synth_seq(6, 10, 78))}
    # weights and inputs are reproducible from their seeds (oracle: init_weights / synth_seq): only checksums are stored
    torch.save({"weight_checksums": {k: S.checksum(v) for k, v in net.state_dict().items()}, "seq_checksum": S.checksum(seq),
                "matrix": out, "seed_w": 1234, "seed_x": 77, "merges": merges, "probe": probe},
               os.path.join(HERE, "ssp_small.pt"))
    print("wrote ssp_small.pt", tuple(out.shape), len(merges), "merges")


if __name__ == "__main__":
    main()
