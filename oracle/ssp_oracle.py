"""CPU oracle for the R-level SSP step of the eval pre-step (SURVEY.md 8 f2) — TEST INFRASTRUCTURE ONLY.

Restates, with an explicit weight dict and torch CPU ops in the reference's order:
  * SinkhornNet.forward                 /root/reference/models/sinkhorn_network.py:39-51   (MLP -> tanh logits)
  * SinkhornNet.sinkhorn                /root/reference/models/sinkhorn_network.py:30-37   (exp(x / tau), n_iters x column / row normalisation)
  * the assignment post-processing      /root/reference/coco_scripts/eval_coco.py:184-200  (transpose -> Munkres on the profit
    matrix -> column assigned to each of the first n rows -> argsort -> positions of a repeated role's slots)
  * verb_rank_merge                     /root/reference/utils/tools.py:35-71
Only tests/ may import this module; the product path (vsr-guided-cic_b200/) never does.

Pin: tests/golden/ssp_small.pt is generated from the UNMODIFIED reference classes/functions imported from
/root/reference (tests/golden/make_golden_ssp.py); tests/test_oracle_ssp.py checks this oracle against it bit for bit
(matrix) and exactly (merges).  The reference calls munkres==1.0.12 (vsr.yml:211), which is absent from this image: an
optimal assignment of a profit matrix is unique unless two assignments tie exactly, so the pin for that step is
scipy.optimize.linear_sum_assignment(maximize=True) on the same matrix (float Sinkhorn outputs: no exact ties)."""
from typing import Dict, List, Sequence

import numpy as np
import torch
import torch.nn.functional as F

PARAMS = ("W1_txt.weight", "W1_txt.bias", "W1_vis.weight", "W1_vis.bias", "W2_vis.weight", "W2_vis.bias",
          "W_fc_pos.weight", "W_fc_pos.bias", "W_fc.weight", "W_fc.bias")     # state_dict order (sinkhorn_network.py:11-15)


def init_weights(N: int = 10, seed: int = 1234) -> Dict[str, torch.Tensor]:
    """Same initialisers in the same order as SinkhornNet.__init__ + init_weights (sinkhorn_network.py:11-28)."""
    torch.manual_seed(seed)
    from torch import nn
    layers = [("W1_txt", nn.Linear(300, 128)), ("W1_vis", nn.Linear(2048, 512)), ("W2_vis", nn.Linear(512, 128)),
              ("W_fc_pos", nn.Linear(260, 256)), ("W_fc", nn.Linear(256, N))]
    W = {}
    for name, lin in layers:
        nn.init.xavier_normal_(lin.weight)
        nn.init.constant_(lin.bias, 0)
        W[name + ".weight"], W[name + ".bias"] = lin.weight.detach().clone(), lin.bias.detach().clone()
    return W


def synth_seq(b: int = 6, N: int = 10, seed: int = 77) -> torch.Tensor:
    """Synthetic (b, N, 2352) role-slot rows: relu(randn) features, position features in [0, 1], and two problems whose
    trailing rows are zero padding (a role held by fewer than N slots, eval_coco.py:178-182)."""
    g = torch.Generator().manual_seed(seed)
    seq = torch.relu(torch.randn((b, N, 2352), generator=g))
    seq[:, :, 2348:] = torch.rand((b, N, 4), generator=g)
    if b > 2:
        seq[1, 4:] = 0
        seq[2, 2:] = 0
    return seq


def checksum(t: torch.Tensor) -> float:
    """sum_i t_i * ((i + 1) mod 97) in float64, summed pairwise with elementwise adds.  Each add is one IEEE rounding, so
    the value is the same on every host; torch.sum's order, and with it the last bits, depends on the CPU's vector width."""
    t = t.double().flatten()
    x = t * torch.arange(1, t.numel() + 1, dtype=torch.float64).remainder(97.0)
    while x.numel() > 1:
        if x.numel() % 2:
            x = torch.cat([x, x.new_zeros(1)])
        x = x[0::2] + x[1::2]
    return float(x.sum())


def logits(W, seq: torch.Tensor) -> torch.Tensor:
    """(B, N, 2352) -> tanh logits (B, N, N)   sinkhorn_network.py:39-49"""
    x_txt, x_vis, x_pos = seq[:, :, :300], seq[:, :, 300:2348], seq[:, :, 2348:]
    x_txt = F.relu(F.linear(x_txt, W["W1_txt.weight"], W["W1_txt.bias"]))
    x_vis = F.relu(F.linear(x_vis, W["W1_vis.weight"], W["W1_vis.bias"]))
    x_vis = F.relu(F.linear(x_vis, W["W2_vis.weight"], W["W2_vis.bias"]))
    x = torch.cat((x_txt, x_vis, x_pos), dim=-1)
    x = F.relu(F.linear(x, W["W_fc_pos.weight"], W["W_fc_pos.bias"]))
    return torch.tanh(F.linear(x, W["W_fc.weight"], W["W_fc.bias"]))


def sinkhorn(x: torch.Tensor, n_iters: int = 20, tau: float = 0.1) -> torch.Tensor:
    """sinkhorn_network.py:30-37 (note the reference's epsilon 10e-8 = 1e-7)."""
    x = torch.exp(x / tau)
    for _ in range(n_iters):
        x = x / (10e-8 + torch.sum(x, -2, keepdim=True))
        x = x / (10e-8 + torch.sum(x, -1, keepdim=True))
    return x


def forward(W, seq: torch.Tensor, n_iters: int = 20, tau: float = 0.1) -> torch.Tensor:
    return sinkhorn(logits(W, seq), n_iters, tau)


def assign(matrix: torch.Tensor) -> np.ndarray:
    """Optimal assignment of the TRANSPOSED doubly-stochastic matrix as eval_coco.py:187-189 computes it
    (munkres on make_cost_matrix(mx) = maximise the profit mx): returns col[r] for every row r of mx = matrix^T."""
    from scipy.optimize import linear_sum_assignment
    mx = matrix.detach().cpu().double().numpy().T
    rows, cols = linear_sum_assignment(mx, maximize=True)
    out = np.zeros(mx.shape[0], dtype=np.int64)
    out[rows] = cols
    return out


def region_order(matrix: torch.Tensor, slots: Sequence[int]) -> List[int]:
    """eval_coco.py:190-200: the slots (positions in the caption's slot list) that hold one repeated role, re-ordered by
    the assignment: sr_re[i] = column assigned to row i (i < len(slots)); order = argsort(sr_re); result[j] = slots[order[j]]."""
    a = assign(matrix)
    sr_re = np.array([a[i] for i in range(len(slots))])
    order = np.argsort(sr_re)
    return [slots[int(i)] for i in order]


def verb_rank_merge(la: List[int], lb: List[int]) -> List[int]:
    """utils/tools.py:35-71: merge the slot order of a second verb (lb) into the first (la).  Slots both lists contain keep
    la's relative order (lb is rewritten in place to agree); every slot only in lb is inserted in front of the next shared
    slot to its right in lb, or appended when there is none."""
    la, lb = list(la), list(lb)
    merged = list(la)
    same, pos_in_b = [], []
    for a in la:
        for j, b in enumerate(lb):
            if a == b:
                same.append(a)
                pos_in_b.append(j)
                break
    if pos_in_b != sorted(pos_in_b):
        for j, p in enumerate(sorted(pos_in_b)):
            lb[p] = same[j]
    right, right_of = None, {}
    for b in reversed(lb):
        if b not in same:
            right_of[b] = right
        else:
            right = b
    for b in lb:
        if b not in same:
            r = right_of[b]
            if r is None:
                merged.append(b)
            else:
                for j, m in enumerate(merged):
                    if m == r:
                        merged.insert(j, b)
                        break
    return merged
