"""A/B timing of the decoder's LSTM CTA forms selected with las_debug_set_option(5, v), interleaved on the same box.

    python tools/decoder_ab.py 0 1 [0 1 ...]      # 0 = weights-stationary form (default), 1 = shared-memory operands
"""
import os
import sys

import torch

ROOT = os.environ.get("LAS_ROOT") or os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402


def main():
    lib = _cabi.load_library()
    flags = [int(a) for a in sys.argv[1:]] or [0]
    cfgname, B, T, S = "paper", 64, 1600, 300
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
    enc = las.listener(x.cuda())
    res = {f: [] for f in flags}
    outs = {}
    for f in flags:  # same sums in the same order per output: every variant must be bit-identical to the first
        _cabi.check(lib.las_debug_set_option(5, f))
        pred, _ = las.speller(enc, None, 0.0)
        outs[f] = (torch.stack(pred).clone(), las.speller.last_tokens.clone())
    for f in flags[1:]:
        print(f"flags={f} vs flags={flags[0]}: bit-identical={all(torch.equal(a, b) for a, b in zip(outs[f], outs[flags[0]]))}")
    for rep in range(4):
        for f in flags:
            lib.las_debug_set_option(5, f)
            las.speller(enc, None, 0.0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                las.speller(enc, None, 0.0)
            e1.record()
            torch.cuda.synchronize()
            res[f].append(e0.elapsed_time(e1) / 5 / S * 1e3)
    lib.las_debug_set_option(5, 0)
    for f in flags:
        v = sorted(res[f])
        print(f"flags={f}: us/step median {v[len(v) // 2]:.3f}  min {v[0]:.3f}  max {v[-1]:.3f}")


if __name__ == "__main__":
    main()
