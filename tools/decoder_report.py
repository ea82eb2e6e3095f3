"""Decoder-only timing + cross-role timeline (globaltimer) on the GPU."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402


def main():
    lib = _cabi.load_library()
    cfgname, B, T, S = "paper", 64, 1600, 300
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
    enc = las.listener(x.cuda())
    for _ in range(2):
        las.speller(enc, None, 0.0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        las.speller(enc, None, 0.0)
    e1.record()
    torch.cuda.synchronize()
    print(f"speller c3 bf16: {e0.elapsed_time(e1) / 3:.3f} ms  ({e0.elapsed_time(e1) / 3 / S * 1e3:.2f} us/step)")
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    buf = torch.zeros(512 + 5 * 32 * 8 + 8 * n_sm, dtype=torch.int64, device="cuda")  # include/las_b200.h las_debug_set_trace
    lib.las_debug_set_trace(_cabi.ptr(buf))
    las.speller(enc, None, 0.0)
    torch.cuda.synchronize()
    lib.las_debug_set_trace(None)
    raw = buf.cpu().numpy()
    t = raw[512:512 + 5 * 32 * 8].reshape(5, 32, 8)
    allc = raw[512 + 5 * 32 * 8:].reshape(n_sm, 8)
    names = [["in ready", "tma issued", "mma issued", "tmem_full", "stored", "signalled", "h-part mma", "-"],
             ["in ready", "tma issued", "mma issued", "tmem_full", "stored", "signalled", "h-part mma", "-"],
             ["h arrived", "q", "softmax", "ctx mma", "ctx published", "logits", "word published", "-"]]
    for s in range(4, 9):
        base = t[0, s, 0]
        print(f"step {s} (ns relative to layer-0 'input ready'):")
        for role, rn in enumerate(["L0 cta0", "L1 cta0", "att cta0"]):
            print(f"   {rn}: " + "  ".join(f"{names[role][i]}={int(t[role, s, i] - base)}" for i in range(7)))
        print(f"   next step L0 input ready at +{int(t[0, s + 1, 0] - base)} ns")
        print("   att fine (rel. h arrived): " + "  ".join(f"{n}={int(t[3, s, i] - t[3, s, 0])}" for i, n in enumerate(
            ["h", "dot", "shfl", "q sync", "energy", "max sync", "sum sync"])))
        print(f"   L0 epilogue: word column gathered at +{int(t[4, s, 1] - base)} ns")
        print(f"   L0 producer: elected at +{int(t[4, s, 0] - base)} ns, TMA instruction issued at +{int(t[4, s, 2] - base)} ns")
        print(f"   critical activation part (ns): L0 fenced={int(t[4, s, 6] - base)} landed={int(t[4, s, 3] - base)}  "
              f"L1 fenced={int(t[4, s, 7] - base)} landed={int(t[4, s, 5] - base)}")
        if s == 8:
            spread(allc, base)
        print(f"   attention CTA 0: {int(t[2, s + 1, 7] - t[2, s, 7])} SM cycles in {int(t[2, s + 1, 0] - t[2, s, 0])} ns "
              f"-> {1e3 * (t[2, s + 1, 7] - t[2, s, 7]) / max(1, (t[2, s + 1, 0] - t[2, s, 0])):.0f} MHz")


def spread(allc, base):
    """Step 8, every CTA: min / max of each stamp relative to layer-0 CTA 0's 'input ready'."""
    def mm(rows, slot):
        v = allc[rows, slot] - base
        return f"{int(v.min())}..{int(v.max())}"
    print("step 8 spread over CTAs (ns, min..max):")
    for name, rows in (("L0", slice(0, 32)), ("L1", slice(32, 64))):
        print(f"   {name}: in ready {mm(rows, 0)}  tmem_full {mm(rows, 1)}  stored {mm(rows, 2)}  signalled {mm(rows, 3)}")
    rows = slice(64, 128)
    print(f"   att: h arrived {mm(rows, 0)}  softmax {mm(rows, 1)}  ctx published {mm(rows, 3)}")


if __name__ == "__main__":
    main()
