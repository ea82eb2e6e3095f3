"""Times the generic tensor-core decoder step (csrc/gen_step.cu) on the reference's shipped config: speller 1024x2 on a synthetic
encoder output.  usage: python tools/gen_step_probe.py [B] [S] [U]   (LAS_PROBE_OPTS="12=0,13=4" sets debug options first)"""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
S = int(sys.argv[2]) if len(sys.argv) > 2 else 64
U = int(sys.argv[3]) if len(sys.argv) > 3 else 200
lib = _cabi.load_library()
for kv in filter(None, os.environ.get("LAS_PROBE_OPTS", "").split(",")):
    k, v = kv.split("=")
    _cabi.check(lib.las_debug_set_option(int(k), int(v)))
c = tl.CONFIGS["shipped"]
las = tl.build_model("shipped", max_label_len=S, seed=17, gain=3.0, precision=os.environ.get("LAS_PROBE_PRECISION", "bf16")).cuda()
g = torch.Generator().manual_seed(1)
enc = torch.tanh(torch.randn(B, U, 2 * c["H"], generator=g)).cuda()
for _ in range(2):
    las.speller(enc, None, 0.0)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
reps = int(os.environ.get("LAS_PROBE_REPS", "5"))
e0.record()
for _ in range(reps):
    las.speller(enc, None, 0.0)
e1.record()
torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / reps
print(f"B={B} S={S} U={U}: {ms:.3f} ms per decode, {1000 * ms / S:.2f} us per step (includes the per-call psi GEMM and prologue)")
if os.environ.get("LAS_PROBE_TRACE"):
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    buf = torch.zeros(512 + 5 * 32 * 8 + 8 * n_sm, dtype=torch.int64, device="cuda")  # include/las_b200.h las_debug_set_trace
    lib.las_debug_set_trace(_cabi.ptr(buf))
    las.speller(enc, None, 0.0)
    torch.cuda.synchronize()
    lib.las_debug_set_trace(None)
    t = buf.cpu().numpy()
    names = {0: ("attention", ["start", "dep ok", "q+sync1", "energies+softmax", "partial ctx", "sync2", "combine", "logits", "sync3", "tail"]),
             1: ("layer 0", ["start", "setup", "indep issued", "dep ok", "mma done", "staged", "cells", "first dependent stage landed", "last mma issued"]),
             2: ("layer 1", ["start", "setup", "indep issued", "dep ok", "mma done", "staged", "cells", "first dependent stage landed", "last mma issued"])}
    for slot, (nm, labels) in names.items():
        v = t[16 * slot:16 * slot + len(labels)]
        print(nm, " ".join(f"{labels[i]}:{(v[i] - v[0]) / 1.965e3:.2f}" for i in range(len(labels))), "(us from the CTA's start, last step)")
    g = lambda slot, i: int(t[16 * slot + i])
    print(f"globaltimer chain (us): attention dep_ok -> end {(g(0, 11) - g(0, 10)) / 1e3:.2f} | -> layer 0 dep_ok {(g(1, 10) - g(0, 11)) / 1e3:.2f} | "
          f"layer 0 dep_ok -> end {(g(1, 11) - g(1, 10)) / 1e3:.2f} | -> layer 1 dep_ok {(g(2, 10) - g(1, 11)) / 1e3:.2f} | "
          f"layer 1 dep_ok -> end {(g(2, 11) - g(2, 10)) / 1e3:.2f}   (last step: the attention stamps are one kernel later than the layers')")
    if os.environ.get("LAS_PROBE_TRACE") == "2":
        v = t[16:16 + 160]
        print("layer 0 producer: (after weights issue, after acts issue) per stage, us:", " ".join(f"({(v[48 + 2 * i] - v[0]) / 1.965e3:.2f},{(v[49 + 2 * i] - v[0]) / 1.965e3:.2f})" for i in range(17)))
        print("layer 0 consumer: stage landed, us:", " ".join(f"{(v[100 + i] - v[0]) / 1.965e3:.2f}" for i in range(17)))
