"""A/B of one las_debug_set_option on a bench workload shape: LAS.forward outputs compared bit for bit, decoder timed both ways.
usage: python tools/option_ab.py KEY VALUE [config] [B] [T] [S]     (default: paper 64 1600 300 = workload c3)"""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402

key, val = int(sys.argv[1]), int(sys.argv[2])
cfg = sys.argv[3] if len(sys.argv) > 3 else "paper"
B = int(sys.argv[4]) if len(sys.argv) > 4 else 64
T = int(sys.argv[5]) if len(sys.argv) > 5 else 1600
S = int(sys.argv[6]) if len(sys.argv) > 6 else 300
lib = _cabi.load_library()
c = tl.CONFIGS[cfg]
las = tl.build_model(cfg, max_label_len=S, seed=17, gain=3.0, precision=os.environ.get("LAS_AB_PRECISION", "bf16")).cuda()
x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
x = x.cuda()
enc = las.listener(x)


def run():
    for _ in range(2):
        preds, attns = las.speller(enc, None, 0.0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        preds, attns = las.speller(enc, None, 0.0)
    e1.record()
    torch.cuda.synchronize()
    tf, _ = las.speller(enc, labels.cuda(), 1.1)
    return torch.stack(preds).clone(), torch.stack([a[0] for a in attns]).clone(), torch.stack(tf).clone(), e0.elapsed_time(e1) / 5


base = run()
_cabi.check(lib.las_debug_set_option(key, val))
alt = run()
same = all(bool(torch.equal(a, b)) for a, b in zip(base[:3], alt[:3]))
print(f"{cfg} B={B} T={T} S={S}: option {key}={val}: {alt[3]:.3f} ms per decode = {1000 * alt[3] / S:.2f} us/step "
      f"(default {base[3]:.3f} ms = {1000 * base[3] / S:.2f} us/step); greedy log-probs, attention, teacher-forced log-probs bit-identical: {same}")
