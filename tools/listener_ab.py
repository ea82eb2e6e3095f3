"""A/B timing of listener variants: python tools/listener_ab.py key=value[,key=value] ...  (las_debug_set_option pairs per variant)"""
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
    variants = [dict((int(k), int(v)) for k, v in (kv.split("=") for kv in a.split(","))) for a in sys.argv[1:]] or [{}]
    c = tl.CONFIGS["paper"]
    x, _ = tl.make_inputs(64, 1600, c["F"], 4, c["V"], seed=17)
    lis = tl.build_model("paper", max_label_len=4, seed=17, gain=3.0, precision="bf16").listener.cuda()
    x = x.cuda()
    res = [[] for _ in variants]
    outs = []
    for v in variants:  # outputs of every variant against the first one
        for k, val in v.items():
            _cabi.check(lib.las_debug_set_option(k, val))
        outs.append(lis(x).clone())
    for v, o in zip(variants[1:], outs[1:]):
        print(f"{v} vs {variants[0]}: max-abs diff {float((o - outs[0]).abs().max()):.3e}  bit-identical={torch.equal(o, outs[0])}")
    for rep in range(4):
        for i, v in enumerate(variants):
            for k, val in v.items():
                lib.las_debug_set_option(k, val)
            lis(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                lis(x)
            e1.record()
            torch.cuda.synchronize()
            res[i].append(e0.elapsed_time(e1) / 5)
    for i, v in enumerate(variants):
        r = sorted(res[i])
        print(f"{v}: listener ms median {r[len(r) // 2]:.4f}  min {r[0]:.4f}  max {r[-1]:.4f}")


if __name__ == "__main__":
    main()
