"""Listener-only report on the GPU: bf16 path vs fp32 path vs golden, plus per-phase device times."""
import ctypes
import glob
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402
from las_pytorch_b200 import _cabi  # noqa: E402


def phases(lib):
    buf = ctypes.create_string_buffer(1 << 20)
    _cabi.check(lib.las_prof_report(buf, len(buf)))
    out = {}
    for line in buf.value.decode().splitlines():
        name, t, n = line.rsplit(" ", 2)
        out[name] = out.get(name, 0.0) + float(t)
    return out


def main():
    lib = _cabi.load_library()
    for name in tl.golden_cases():
        g = tl.load_golden(name)
        cfg = str(g["cfg"])
        if cfg in ("tiny_mh", "tiny_nomlp", "tiny_gru", "tiny_rnn"):  # attention variants run in the fp32 mode only
            continue
        las = tl.build_model(cfg, max_label_len=4, seed=int(g["seed"]), gain=float(g["gain"]), precision="bf16")
        sd = {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
        if sd:
            las.load_state_dict(sd)
        lis = las.listener.cuda()
        enc = lis(torch.from_numpy(g["x"]).cuda())
        torch.cuda.synchronize()
        err = float(np.abs(enc.cpu().numpy() - g["enc_f64"]).max())
        print(f"{name + '.npz':24s} bf16 listener max-abs err vs fp64 reference = {err:.3e}", flush=True)
    for cfgname, B, T in (("paper", 64, 1600), ("small", 32, 1600), ("paper", 16, 3000)):
        c = tl.CONFIGS[cfgname]
        x, _ = tl.make_inputs(B, T, c["F"], 4, c["V"], seed=17)
        x = x.cuda()
        outs = {}
        for prec in ("fp32", "bf16"):
            las = tl.build_model(cfgname, max_label_len=4, seed=17, gain=3.0, precision=prec)
            lis = las.listener.cuda()
            for _ in range(2):
                outs[prec] = lis(x)
            torch.cuda.synchronize()
            lib.las_prof_enable(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                lis(x)
            e1.record()
            torch.cuda.synchronize()
            ph = {k: round(v / 3, 4) for k, v in phases(lib).items()}
            lib.las_prof_enable(0)
            print(f"{cfgname} B={B} T={T} {prec}: {e0.elapsed_time(e1) / 3:.3f} ms/listener  phases(ms)={ph}", flush=True)
        d = (outs["bf16"] - outs["fp32"]).abs()
        print(f"   bf16 vs fp32 listener: max {float(d.max()):.3e} mean {float(d.mean()):.3e}", flush=True)


if __name__ == "__main__" and len(sys.argv) == 1:
    main()


def trace():
    lib = _cabi.load_library()
    c = tl.CONFIGS["paper"]
    x, _ = tl.make_inputs(64, 1600, c["F"], 4, c["V"], seed=17)
    lis = tl.build_model("paper", max_label_len=4, seed=17, gain=3.0, precision="bf16").listener.cuda()
    x = x.cuda()
    import sys as _s
    opt = int(_s.argv[2]) if len(_s.argv) > 2 else 1
    lib.las_debug_set_option(1, opt)
    nacc = int(_s.argv[3]) if len(_s.argv) > 3 else 0
    lib.las_debug_set_option(4, nacc)
    if len(_s.argv) > 4:  # utterances per recurrence cluster (16 / 32 / 64): 64 is the form that runs under the decoder
        lib.las_debug_set_option(9, int(_s.argv[4]))
    print(f"recurrence A operand in TMEM: {opt}; accumulators: {nacc or 'default'}")
    ref = tl.build_model("paper", max_label_len=4, seed=17, gain=3.0, precision="fp32").listener.cuda()(x)
    out = lis(x)
    print(f"bf16 vs fp32 listener max err {float((out - ref).abs().max()):.3e}")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        lis(x)
    e1.record()
    torch.cuda.synchronize()
    print(f"listener c3 bf16: {e0.elapsed_time(e1) / 5:.3f} ms")
    buf = torch.zeros(64 * 8, dtype=torch.int64, device="cuda")
    lib.las_debug_set_trace(_cabi.ptr(buf))
    lis(x)
    torch.cuda.synchronize()
    lib.las_debug_set_trace(None)
    t = buf.cpu().numpy().reshape(64, 8)
    names = ["h_full ok", "mma issued", "mma_done ok", "tmem ld", "gates", "gstores", "staged+fence", "bulk issued"]
    print("recurrence trace (cycles relative to 'h_full ok' of each step; CTA 0):")
    for s in range(2, 12):
        base = t[s, 0]
        print(f"  step {s:2d}: " + "  ".join(f"{n}={int(t[s, i] - base):5d}" for i, n in enumerate(names)) +
              f"   | next h_full ok at +{int(t[s + 1, 0] - base)}")


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "trace":
    trace()
