"""The R-level SSP oracle (oracle/ssp_oracle.py) against golden vectors of the unmodified reference (CPU)."""
import os

import torch

from oracle import ssp_oracle as S

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ssp_small.pt")


def test_sinkhorn_oracle_matches_reference_golden():
    fx = torch.load(GOLD, weights_only=False)
    W = S.init_weights(10, fx["seed_w"])
    for k, c in fx["weight_checksums"].items():
        assert S.checksum(W[k]) == c, k                     # same RNG stream as the reference's constructor
    seq = S.synth_seq(6, 10, fx["seed_x"])
    assert S.checksum(seq) == fx["seq_checksum"]
    with torch.no_grad():
        out = S.forward(W, seq)
        probe = S.forward(W, S.synth_seq(6, 10, fx["probe"]["seed_x"]))
    if torch.equal(probe, fx["probe"]["matrix"]):
        # this host's float32 CPU kernels round like those of the host that made the golden vectors
        assert torch.equal(out, fx["matrix"])               # bit for bit
    else:
        # other BLAS / vector-width paths reorder the sums; exp(x / 0.1) and 20 normalisation rounds amplify that to
        # ~110 ulps (1.3e-5 relative) at most over the code paths measured
        assert torch.allclose(out, fx["matrix"], rtol=5e-5, atol=0)
    # the matrix is (nearly) doubly stochastic and its optimal assignment is a permutation
    assert torch.allclose(out.sum(-1), torch.ones(6, 10), atol=1e-4)
    for i in range(6):
        a = S.assign(out[i])
        assert sorted(a.tolist()) == list(range(10))


def test_verb_rank_merge_matches_reference_golden():
    fx = torch.load(GOLD, weights_only=False)
    for la, lb, want in fx["merges"]:
        assert S.verb_rank_merge(la, lb) == want, (la, lb)


def test_region_order_is_a_permutation_of_the_slots():
    fx = torch.load(GOLD, weights_only=False)
    slots = [7, 2, 5, 3]
    order = S.region_order(fx["matrix"][1], slots)
    assert sorted(order) == sorted(slots)
