"""Shared test helpers: model configs, seeded synthetic weights / inputs (SURVEY.md section 8d)."""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def golden_cases():
    """Names of the model-forward golden cases (tests/golden/<name>.npz); the `ref_*` files are the solver / checkpoint fixtures."""
    import glob

    return sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")) if not os.path.basename(p).startswith("ref_"))


def load_golden(name):
    """tests/golden/<name>.npz as a dict of arrays.  A case whose weights are reproduced from the seed may be stored compactly
    (tests/golden/make_golden.py `compact`) to keep the file under 1 MB: its input `x` is then regenerated from the seed as
    well (checked by SHA-256), and an fp64 output may be stored as a float32 difference from the fp32 one.  That restores
    the fp64 output to within 1e-13, below the tightest tolerance any test applies to it (1e-12)."""
    import hashlib

    g = dict(np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False))
    if "x" not in g:
        c = CONFIGS[str(g["cfg"])]
        B, T, _ = (int(n) for n in g["x_shape"])
        x, labels = make_inputs(B, T, c["F"], g["labels"].shape[1], c["V"], seed=int(g["seed"]))
        x = x.numpy()
        assert hashlib.sha256(x.tobytes()).hexdigest() == str(g["x_sha256"]), f"{name}: seeded input differs from the golden run's"
        assert np.array_equal(labels.numpy(), g["labels"])
        g["x"] = x
    for k in ("enc", "logp", "attn"):
        if f"{k}_f64" not in g:
            g[f"{k}_f64"] = g[f"{k}_f32"].astype(np.float64) + g.pop(f"{k}_f64_minus_f32")
    return g


# name -> (listener kwargs, speller kwargs).  V=30, D=64 from config/librispeech-config.yaml:12,31.
CONFIGS = {
    # tiny shapes whose weights are stored inside the golden files
    "tiny": dict(F=40, H=16, L=2, sl=2, V=30, D=16),
    "odd": dict(F=40, H=24, L=3, sl=3, V=42, D=20),   # V+E not a multiple of 8, 3 speller layers (common_voice-like V)
    # Speller / Attention variants of SURVEY.md section 8 row f4 (fp32 mode): two heads + dim_reduce; no MLP in the attention
    "tiny_mh": dict(F=40, H=16, L=2, sl=2, V=30, D=16, heads=2),
    "tiny_nomlp": dict(F=40, H=16, L=2, sl=2, V=30, D=16, use_mlp=False),
    # rnn_unit variants (the reference resolves the string with getattr(nn, rnn_unit.upper()), model/las_model.py:69,156)
    "tiny_gru": dict(F=40, H=16, L=2, sl=2, V=30, D=16, unit="GRU"),
    "tiny_rnn": dict(F=40, H=16, L=2, sl=2, V=30, D=16, unit="RNN"),
    # README small LAS (listener 128x2, speller 256x2) and the paper-size model
    "small": dict(F=40, H=128, L=2, sl=2, V=30, D=64),
    "paper": dict(F=40, H=256, L=3, sl=2, V=30, D=64),
    # the reference's shipped config (config/librispeech-config.yaml:13-34): listener 512x3, speller 1024x2
    "shipped": dict(F=40, H=512, L=3, sl=2, V=30, D=64),
}


def build_model(cfg, max_label_len, decode_mode=1, seed=17, gain=1.0, precision="fp32", module=None):
    """Construct (listener, speller, las) under torch.manual_seed(seed), then scale every 2-D parameter by `gain`
    (the "gain-3" ladder of SURVEY.md A.6).  `module` = the module providing Listener/Speller/LAS (ours by default).
    The optional config key `activate` is the attention MLP's activation ("relu", the default, or "None")."""
    if module is None:
        import las_pytorch_b200 as module
    c = CONFIGS[cfg] if isinstance(cfg, str) else cfg
    torch.manual_seed(seed)
    extra = {} if module.__name__.startswith("model") else {"precision": precision}
    unit = c.get("unit", "LSTM")
    listener = module.Listener(input_feature_dim=c["F"], hidden_size=c["H"], num_layers=c["L"], rnn_unit=unit,
                               use_gpu=False, **extra)
    speller = module.Speller(vocab_size=c["V"], hidden_size=2 * c["H"], rnn_unit=unit, num_layers=c["sl"],
                             max_label_len=max_label_len, use_mlp_in_attention=c.get("use_mlp", True), mlp_dim_in_attention=c["D"],
                             mlp_activate_in_attention=c.get("activate", "relu"), listener_hidden_size=c["H"], multi_head=c.get("heads", 1),
                             decode_mode=decode_mode, use_gpu=False, **extra)
    las = module.LAS(listener, speller)
    if gain != 1.0:
        with torch.no_grad():
            for p in las.parameters():
                if p.dim() == 2:
                    p.mul_(gain)
    return las


def state_dict_numpy(las):
    return {k: v.detach().cpu().numpy() for k, v in las.state_dict().items()}


def make_inputs(B, T, F, S, V, seed=17, pad_tail=0):
    """x = randn(B,T,F) under a seeded generator; labels randint(2,V) as indices [B,S] (0=<sos>/PAD, 1=<eos>)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, F, generator=g)
    if pad_tail:
        x[:, T - pad_tail:, :] = 0.0  # zero padding as utils/data.py:132 does
    labels = torch.randint(2, V, (B, S), generator=g)
    return x, labels


def onehot(labels, V):
    return torch.nn.functional.one_hot(labels, V).to(torch.int64)


def weights_fingerprint(sd):
    """Order-independent fingerprint of a state dict (used to prove seeded weights match the golden run)."""
    tot = 0.0
    for k in sorted(sd):
        a = np.asarray(sd[k], dtype=np.float64)
        tot += float(a.sum()) * 1.0 + float((a * a).sum()) * 3.0 + float(np.abs(a).max()) * 7.0
    return tot
