"""A/B of the attention split (las_debug_set_option(11, v)): decoder us/step per workload shape.
    python tools/split_ab.py c2|c3|c4 v1 v2 ...      # 1 = split long encoders over two CTAs (default), 0 = never"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402

SH = {"c2": ("small", 32, 1600, 300), "c3": ("paper", 64, 1600, 300), "c4": ("paper", 16, 3000, 600)}
lib = _cabi.load_library()
cfgname, B, T, S = SH[sys.argv[1]]
vals = [int(v) for v in sys.argv[2:]]
c = tl.CONFIGS[cfgname]
las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
enc = las.listener(x.cuda())
res = {v: [] for v in vals}
toks = {}
for rep in range(3):
    for v in vals:
        _cabi.check(lib.las_debug_set_option(11, v))
        las.speller(enc, None, 0.0)
        toks[v] = las.speller.last_tokens.clone()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            las.speller(enc, None, 0.0)
        e1.record()
        torch.cuda.synchronize()
        res[v].append(e0.elapsed_time(e1) / 5 / S * 1e3)
lib.las_debug_set_option(11, 1)
for v in vals:
    r = sorted(res[v])
    print(f"{sys.argv[1]} option11={v}: us/step median {r[1]:.3f}  token agreement with option11={vals[0]}: {float((toks[v] == toks[vals[0]]).float().mean()):.4f}")
