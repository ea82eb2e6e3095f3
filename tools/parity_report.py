"""Prints max-abs errors of both precisions against every golden case (diagnostic; numbers quoted in DESIGN.md)."""
import glob
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import las_testlib as tl  # noqa: E402


def main():
    print(f"{'case':18s} {'prec':5s} {'enc':>10s} {'logp':>10s} {'attn':>10s} {'argmax agree':>13s}  (vs the reference's fp64 run)")
    for name in tl.golden_cases():
        g = tl.load_golden(name)
        cfg, mode = str(g["cfg"]), str(g["mode"])
        c = tl.CONFIGS[cfg]
        S = g["logp_f64"].shape[0]
        for prec in ("fp32", "bf16"):
            if prec == "bf16" and (c.get("heads", 1) > 1 or not c.get("use_mlp", True) or c.get("unit", "LSTM") != "LSTM"):
                continue  # attention variants run in the fp32 mode only
            las = tl.build_model(cfg, max_label_len=S, decode_mode=0 if mode == "raw" else 1, seed=int(g["seed"]), gain=float(g["gain"]), precision=prec)
            sd = {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
            if sd:
                las.load_state_dict(sd)
            las = las.cuda()
            x = torch.from_numpy(g["x"]).cuda()
            gt = tl.onehot(torch.from_numpy(g["labels"]).long(), c["V"]).cuda() if mode == "tf" else None
            np.random.seed(0)
            preds, attns = las(x, gt, 1.1 if mode == "tf" else 0.0, is_training=(mode == "tf"))
            enc = las.listener(x).cpu().numpy()
            logp = torch.stack(preds).cpu().numpy()
            attn = (torch.stack([a[0] for a in attns]) if len(attns[0]) == 1 else torch.stack([torch.stack(list(a)) for a in attns])).cpu().numpy()
            agree = (logp.argmax(-1) == g["logp_f64"].argmax(-1)).mean()
            print(f"{name:18s} {prec:5s} {np.abs(enc - g['enc_f64']).max():10.3e} {np.abs(logp - g['logp_f64']).max():10.3e} "
                  f"{np.abs(attn - g['attn_f64']).max():10.3e} {agree:13.3f}", flush=True)


if __name__ == "__main__":
    main()
