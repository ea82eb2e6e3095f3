"""A/B of a debug option of the fused generic decoder step: outputs compared bit for bit, both timed.
usage: python tools/gen_step_ab.py KEY VALUE [B] [S]"""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402

key, val = int(sys.argv[1]), int(sys.argv[2])
B = int(sys.argv[3]) if len(sys.argv) > 3 else 16
S = int(sys.argv[4]) if len(sys.argv) > 4 else 128
lib = _cabi.load_library()
c = tl.CONFIGS["shipped"]
las = tl.build_model("shipped", max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
enc = torch.tanh(torch.randn(B, 200, 2 * c["H"], generator=torch.Generator().manual_seed(1))).cuda()


def run():
    for _ in range(2):
        preds, _ = las.speller(enc, None, 0.0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        preds, _ = las.speller(enc, None, 0.0)
    e1.record()
    torch.cuda.synchronize()
    return torch.stack(preds).clone(), e0.elapsed_time(e1) / 5 * 1000 / S


base, t0 = run()
_cabi.check(lib.las_debug_set_option(key, val))
try:
    alt, t1 = run()
finally:
    pass
print(f"option {key}={val}: {t1:.2f} us/step (default {t0:.2f}); bit-identical: {bool(torch.equal(base, alt))}; "
      f"max abs diff {float((base - alt).abs().max()):.3e}")
