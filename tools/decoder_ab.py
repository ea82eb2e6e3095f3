"""Timing of the persistent decoder on the c3 shape (paper LAS, 64 utterances, U = 200, 300 greedy steps): µs per decoder step.
It takes no option, so the same script times the library of any tree (LAS_ROOT) -- tools/ab_trees.sh alternates trees with it.

    python tools/decoder_ab.py
    LAS_ROOT=/path/to/other/tree python tools/decoder_ab.py
"""
import os
import sys

import torch

ROOT = os.environ.get("LAS_ROOT") or os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402


def main():
    cfgname, B, T, S = "paper", 64, 1600, 300
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
    enc = las.listener(x.cuda())
    res = []
    for rep in range(4):
        las.speller(enc, None, 0.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            las.speller(enc, None, 0.0)
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) / 5 / S * 1e3)
    v = sorted(res)
    print(f"decoder c3: us/step median {v[len(v) // 2]:.3f}  min {v[0]:.3f}  max {v[-1]:.3f}")


if __name__ == "__main__":
    main()
