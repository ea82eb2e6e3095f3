"""Beam-search decoding time on the benchmark's seeded inputs, next to greedy decoding of the same batch.

    python tools/beam_bench.py [--precision bf16] [--reps 3] [--widths 1,4,8] [--workloads c3,yaml] [--early-exit] [--attention]
                               [--eos-bias X]

Workloads (as bench.py builds them: tests/las_testlib.py seeded weights, gain 3, inputs seed 17):
    c3:   paper LAS (listener 256x3, speller 512x2), 64 x 1600 frames, 300 steps
    yaml: the shipped config (listener 512x3, speller 1024x2), 16 x 1600 frames, 576 steps
Prints one JSON line per (workload, beam width): ms per batch of LAS.beam_search (listener + beam decode), the decode alone in ms and
in us per decoder step, audio seconds per second, greedy LAS.forward on the same batch, and the device.  Timing: CUDA events around
each call after one warm-up call, a 256 MiB buffer written between timed calls so that every call starts with a cold L2, the median of
--reps calls.  Needs a CUDA device; there is no CPU fallback.

--early-exit adds the same LAS.beam_search with early_exit=True (checked every 32 steps) and the steps it ran; --attention adds it with
return_attention=True.  The variants are timed in the same process, call by call after the plain one.  The synthetic models rarely emit
<eos>; --eos-bias X adds X to the <eos> logit's bias (character_distribution.bias[1]) so that hypotheses end at a controlled point.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

WORKLOADS = {"c3": dict(cfg="paper", B=64, T=1600, S=300), "yaml": dict(cfg="shipped", B=16, T=1600, S=576)}
FRAME_SEC = 0.01  # 10 ms frame hop


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16", "fp16"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--widths", default="1,4,8")
    ap.add_argument("--workloads", default="c3,yaml")
    ap.add_argument("--early-exit", action="store_true", help="also time early_exit=True and report the steps run")
    ap.add_argument("--attention", action="store_true", help="also time return_attention=True")
    ap.add_argument("--eos-bias", type=float, default=0.0, help="added to the <eos> logit's bias of the benchmark model")
    args = ap.parse_args()

    import numpy as np
    import torch

    import las_testlib as tl

    if not torch.cuda.is_available():
        raise SystemExit("tools/beam_bench.py needs a CUDA device (no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def timed(fn):
        fn()  # warm-up: module loads, packs, workspaces
        ms = []
        for _ in range(args.reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms))

    device = torch.cuda.get_device_name(dev)
    for name in args.workloads.split(","):
        wl = WORKLOADS[name]
        c = tl.CONFIGS[wl["cfg"]]
        B, T, S = wl["B"], wl["T"], wl["S"]
        las = tl.build_model(wl["cfg"], max_label_len=S, seed=17, gain=3.0, precision=args.precision).to(dev)
        with torch.no_grad():
            las.speller.character_distribution.bias[1] += args.eos_bias
        x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
        x = x.to(dev)
        with torch.no_grad():
            enc = las.listener(x)
            greedy_ms = timed(lambda: las(x, None, 0.0, is_training=False))
            for K in (int(k) for k in args.widths.split(",")):
                batch_ms = timed(lambda: las.beam_search(x, beam_width=K, nbest=1))
                decode_ms = timed(lambda: las.speller.beam_search(enc, beam_width=K, nbest=1))
                line = {
                    "workload": name, "precision": args.precision, "B": B, "T": T, "steps": S, "beam": K, "eos_bias": args.eos_bias,
                    "ms_per_batch": round(batch_ms, 3), "decode_ms": round(decode_ms, 3), "us_per_step": round(1e3 * decode_ms / S, 2),
                    "audio_s_per_s": round(B * T * FRAME_SEC / (batch_ms / 1e3), 1),
                    "greedy_forward_ms_per_batch": round(greedy_ms, 3),
                }
                if args.early_exit:
                    line["early_exit_ms_per_batch"] = round(timed(lambda: las.beam_search(x, beam_width=K, nbest=1, early_exit=True)), 3)
                    line["steps_done"] = int(las.speller.last_steps_done.item())
                    r = las.beam_search(x, beam_width=K, nbest=1)
                    line["max_length"] = int(r.lengths.max().item())
                if args.attention:
                    line["attention_ms_per_batch"] = round(timed(lambda: las.beam_search(x, beam_width=K, nbest=1, return_attention=True)), 3)
                line.update(device=device, reps=args.reps)
                print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
