"""CPU probe (no GPU): how much accuracy do cheaper tensor-core operand schemes keep on the decoder's big GEMMs?

Emulates, inside the oracle (tests' CPU restatement of the reference), the rounding of the operands of every weight
GEMM with both dims >= 256, then compares a free-running beam search with the unmodified oracle:
  f16x3     : x_hi*w_hi + x_hi*w_lo + x_lo*w_hi, hi = fp16(x), lo = fp16(x - hi)             (what libvsrdec runs)
  f16+f8x2  : x_hi*w_hi in fp16, the two residual products with e4m3 operands                  (2/3 of the MMA time)
  f16x1     : x_hi*w_hi only                                                                    (1/3)
Activations are brought to 2^13..2^14 by a power of two per call, or, with act_scale, multiplied by that constant as
libvsrdec's activation twins are (ACT_SCALE_F8 in csrc/common.cuh), saturating like the device conversions do.
Usage: python tools/fp8_probe.py [b] [sharpen] [act_scale]"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "vsr-guided-cic_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch  # noqa: E402
import torch.nn.functional as TF  # noqa: E402
from oracle import vsr_oracle as O  # noqa: E402


def pow2_scale(x, top):
    m = float(x.abs().max())
    if m == 0.0:
        return 1.0
    import math
    return 2.0 ** (top - math.ceil(math.log2(m)))


def e4m3(x):
    return x.clamp(-448.0, 448.0).to(torch.float8_e4m3fn).float()     # __NV_SATFINITE


class Emu:
    def __init__(self, mode, act_scale=None):
        self.mode = mode
        self.act_scale = act_scale

    def linear(self, x, w, b=None):
        if self.mode == "exact" or w.dim() != 2 or min(w.shape) < 256:
            return TF.linear(x, w, b)
        sx, sw = pow2_scale(x, 13) if self.act_scale is None else self.act_scale, pow2_scale(w, 13)
        xs, ws = (x * sx).clamp(-65504.0, 65504.0), w * sw
        xh, wh = xs.half().float(), ws.half().float()
        xl, wl = xs - xh, ws - wh
        shp = x.shape[:-1]
        x2 = lambda t: t.reshape(-1, t.shape[-1])
        y = x2(xh) @ wh.t()
        if self.mode == "f16x3":
            y = y + x2(xh) @ wl.half().float().t() + x2(xl.half().float()) @ wh.t()
        elif self.mode == "f16+f8x2":
            y = y + (x2(e4m3(xh / 32)) @ e4m3(wl * 32).t()) + (x2(e4m3(xl * 32)) @ e4m3(wh / 32).t())
        elif self.mode == "f16x1":
            pass
        y = (y / (sx * sw)).reshape(*shp, w.shape[0])
        return y + b if b is not None else y

    def __getattr__(self, name):
        return getattr(TF, name)


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 32
    sharpen = float(sys.argv[2]) if len(sys.argv) > 2 else 0.0
    act_scale = float(sys.argv[3]) if len(sys.argv) > 3 else None
    torch.set_num_threads(os.cpu_count())
    d = O.Dims()
    W = O.init_weights(d, seed=1234)
    if sharpen:
        W["out_fc.weight"] = W["out_fc.weight"] * sharpen
    statics = O.synth_inputs(b, 50, 10, 20, 2048, seed=1002, vocab_size=d.vocab_size, n_det_range=(10, 50),
                             verb_slots=(2,), verb_vocab_id=17)
    res = {}
    for mode in ("exact", "f16x3", "f16+f8x2", "f16x1"):
        O.F = Emu(mode, act_scale)
        with torch.no_grad():
            outs, lps = O.beam_search(W, d, statics, [3, -1], 5, 1, use_verbs=True, gt=True)
        res[mode] = (outs, lps)
        if mode != "exact":
            ro, rl = res["exact"]
            same = ((outs[0] == ro[0]).all(-1) & (outs[1] == ro[1]).all(-1))
            tok = float((outs[0] == ro[0]).float().mean())
            sel = same.reshape(-1)
            dl = float((lps[0].reshape(b, -1)[sel] - rl[0].reshape(b, -1)[sel]).abs().max()) if sel.any() else float("nan")
            dg = float((lps[1].reshape(b, -1)[sel] - rl[1].reshape(b, -1)[sel]).abs().max()) if sel.any() else float("nan")
            print(f"b={b} sharpen={sharpen} act_scale={act_scale} {mode:9s}: captions identical {int(same.sum())}/{b}, tokens {tok:.4f}, "
                  f"max |dlogp| word {dl:.2e} gate {dg:.2e} (on identical captions)", flush=True)
    O.F = TF


if __name__ == "__main__":
    main()
