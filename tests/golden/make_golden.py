"""Generates tests/golden/*.npz by running the UNMODIFIED reference (a checkout of jiwidi/las-pytorch) on CPU:

    LAS_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py

The reference is imported as-is; only three data-prep-only third-party modules that `utils/functions.py`
imports at module top level are stubbed (SURVEY.md B.1) -- none is reachable from any `forward`.
Each case stores inputs, (for the tiny configs) the full state_dict, and the reference's fp32 and fp64 outputs.
For the larger configs the weights are reproduced from the seed by `las_pytorch_b200`'s own parameter
containers; this script asserts that those are bit-identical to the reference's freshly constructed weights and
stores a fingerprint.  Those cases are stored compactly (`compact`) so that every file stays under 1 MB;
tests/las_testlib.py `load_golden` restores them.
"""
from __future__ import annotations

import copy
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)


def compact(out):
    """Seeded cases: the input is regenerated from the seed (SHA-256 kept to check it), and each fp64 output is kept as a
    float32 difference from the fp32 one where that difference restores it to 1e-13 (not so in the chaotic gain-6 case,
    whose fp32 and fp64 runs are far apart: there the fp64 output is kept as it is)."""
    import hashlib

    x = out.pop("x")
    out["x_shape"] = np.asarray(x.shape, dtype=np.int64)
    out["x_sha256"] = hashlib.sha256(np.ascontiguousarray(x, dtype=np.float32).tobytes()).hexdigest()
    for k in ("enc", "logp", "attn"):
        f32, f64 = out[f"{k}_f32"], out[f"{k}_f64"]
        diff = (f64 - f32).astype(np.float32)
        if np.abs(f32.astype(np.float64) + diff - f64).max() <= 1e-13:
            del out[f"{k}_f64"]
            out[f"{k}_f64_minus_f32"] = diff
    return out


def import_reference():
    ref_root = os.environ.get("LAS_REFERENCE_ROOT")
    if not ref_root:
        raise SystemExit("set LAS_REFERENCE_ROOT to a checkout of the reference (jiwidi/las-pytorch)")
    for name in ("pydub", "editdistance", "python_speech_features"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["pydub"].AudioSegment = object
    sys.modules["python_speech_features"].logfbank = None
    sys.path.insert(0, ref_root)
    import model.las_model as ref  # noqa

    return ref


def run_reference(las, x, gt_onehot, teacher_forced, dtype):
    """Runs the reference LAS on CPU.  Returns enc, logp [S,B,V], attn [S,B,U]."""
    m = copy.deepcopy(las).to(dtype).eval()
    m.speller.float_type = torch.DoubleTensor if dtype == torch.float64 else torch.FloatTensor
    with torch.no_grad():
        enc = m.listener(x.to(dtype))
        if teacher_forced:
            np.random.seed(0)
            preds, attns = m.speller(enc, ground_truth=gt_onehot, teacher_force_rate=1.1)  # always teacher-forced
        else:
            preds, attns = m.speller(enc, ground_truth=None, teacher_force_rate=0)
    logp = torch.stack(preds)
    if len(attns[0]) == 1:
        attn = torch.stack([a[0] for a in attns])                 # [S,B,U]
    else:
        attn = torch.stack([torch.stack(list(a)) for a in attns])  # multi_head > 1: [S,heads,B,U]
    return enc.numpy(), logp.numpy(), attn.numpy()


def make_extras(ref, tl):
    """Fixtures for the "next" rows: (f3) a checkpoint package written by the REFERENCE's own LAS.serialize + torch.save
    (model/las_model.py:42-63, train.py:181-192) together with the reference's outputs for it; (f1) the reference's
    label_smoothing_loss / NLLLoss / LetterErrorRate values (solver/solver.py:11-24,33-45,62,70-92) on seeded inputs."""
    import solver.solver as ref_solver  # the reference's solver (editdistance stubbed: give it a Levenshtein)

    def lev(a, b):
        prev = list(range(len(b) + 1))
        for i, ca in enumerate(a, 1):
            cur = [i]
            for j, cb in enumerate(b, 1):
                cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (ca != cb)))
            prev = cur
        return prev[-1]

    sys.modules["editdistance"].eval = lev
    ref_solver.ed.eval = lev
    # ---- f3: package from the reference
    cfg, B, T, S = "tiny", 3, 32, 8
    c = tl.CONFIGS[cfg]
    ref_las = tl.build_model(cfg, max_label_len=S, decode_mode=1, seed=41, gain=3.0, module=ref)
    opt = torch.optim.Adam(ref_las.parameters(), lr=1e-3)
    pkg = ref_las.serialize(opt, epoch=7, tr_loss=1.25, val_loss=1.5)
    # as nn.DataParallel-wrapped training would have saved it (train.py:76-78): keys carry a "module." prefix in one of the two files
    torch.save(pkg, os.path.join(HERE, "ref_package_tiny.pth.tar"))
    pkg_dp = dict(pkg, state_dict={"module." + k: v for k, v in pkg["state_dict"].items()})
    torch.save(pkg_dp, os.path.join(HERE, "ref_package_tiny_dataparallel.pth.tar"))
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=41)
    gt = tl.onehot(labels, c["V"])
    out = {"x": x.numpy(), "labels": labels.numpy().astype(np.int32)}
    for mode in ("tf", "greedy"):
        enc, logp, attn = run_reference(ref_las, x, gt, mode == "tf", torch.float64)
        out["enc_f64"], out[f"logp_{mode}_f64"], out[f"attn_{mode}_f64"] = enc, logp, attn
    np.savez_compressed(os.path.join(HERE, "ref_package_tiny_outputs.npz"), **out)
    print("ref_package_tiny.pth.tar:", sorted(pkg), "etype =", pkg["etype"])

    # ---- f1: solver losses from the reference's own functions
    g = torch.Generator().manual_seed(43)
    Bs, Ss, V = 5, 12, 30
    logp = torch.log_softmax(3.0 * torch.randn(Bs, Ss, V, generator=g), dim=-1)
    lab = torch.randint(2, V, (Bs, Ss), generator=g)
    lens = torch.tensor([12, 9, 5, 12, 1])
    onehot_zero_pad = tl.onehot(lab, V).float()     # padding rows all zero (what label_smoothing_loss documents)
    lab_pad0 = lab.clone()                           # padding rows = one-hot(0) (what utils/data.py:133-136 produces)
    for b in range(Bs):
        onehot_zero_pad[b, lens[b]:, :] = 0
        lab_pad0[b, lens[b]:] = 0
    onehot_pad0 = tl.onehot(lab_pad0, V).float()
    res = {"logp": logp.numpy(), "labels": lab.numpy().astype(np.int32), "lens": lens.numpy().astype(np.int32)}
    for ls in (0.1, 0.3):
        res[f"ls_zero_pad_{ls}"] = float(ref_solver.label_smoothing_loss(logp, onehot_zero_pad, label_smoothing=ls))
        res[f"ls_pad0_{ls}"] = float(ref_solver.label_smoothing_loss(logp, onehot_pad0, label_smoothing=ls))
    res["nll_ignore0"] = float(torch.nn.NLLLoss(ignore_index=0)(logp.permute(0, 2, 1), lab_pad0))
    res["ler"] = np.asarray(ref_solver.LetterErrorRate(logp.argmax(-1).numpy(), lab_pad0.numpy()), dtype=np.float64)
    np.savez_compressed(os.path.join(HERE, "ref_solver_losses.npz"), **res)
    print("ref_solver_losses.npz:", {k: v for k, v in res.items() if k.startswith(("ls_", "nll"))}, "ler", res["ler"])


def main():
    import las_testlib as tl
    import las_pytorch_b200 as ours

    ref = import_reference()
    if "extras" in sys.argv[1:]:
        make_extras(ref, tl)
        return
    cases = [
        # name, cfg, B, T, S, mode ("tf" | "greedy" | "raw"), gain, store_weights
        ("tiny_tf_g3", "tiny", 3, 32, 6, "tf", 3.0, True),
        ("tiny_greedy_g3", "tiny", 3, 32, 10, "greedy", 3.0, True),
        ("tiny_raw_g3", "tiny", 3, 32, 7, "raw", 3.0, True),
        ("tiny_tf_g1", "tiny", 2, 16, 5, "tf", 1.0, True),
        ("odd_tf_g3", "odd", 2, 48, 9, "tf", 3.0, True),
        ("odd_greedy_g3", "odd", 2, 48, 11, "greedy", 3.0, True),
        ("small_tf_g1", "small", 4, 400, 50, "tf", 1.0, False),   # BASELINE.json configs[0]
        ("small_tf_g3", "small", 4, 400, 50, "tf", 3.0, False),
        ("small_greedy_g3", "small", 4, 400, 40, "greedy", 3.0, False),
        ("small_tf_g6", "small", 2, 160, 30, "tf", 6.0, False),
        ("paper_tf_g3", "paper", 2, 160, 24, "tf", 3.0, False),
        ("paper_greedy_g3", "paper", 2, 160, 24, "greedy", 3.0, False),
        # Speller / Attention variants (SURVEY.md section 8 row f4)
        ("tinymh_tf_g3", "tiny_mh", 3, 32, 6, "tf", 3.0, True),
        ("tinymh_greedy_g3", "tiny_mh", 3, 32, 10, "greedy", 3.0, True),
        ("tinynomlp_tf_g3", "tiny_nomlp", 3, 32, 6, "tf", 3.0, True),
        ("tinynomlp_greedy_g3", "tiny_nomlp", 3, 32, 10, "greedy", 3.0, True),
        ("tinygru_tf_g3", "tiny_gru", 3, 32, 6, "tf", 3.0, True),
        ("tinygru_greedy_g3", "tiny_gru", 3, 32, 10, "greedy", 3.0, True),
        ("tinyrnn_tf_g3", "tiny_rnn", 3, 32, 6, "tf", 3.0, True),
        ("tinyrnn_greedy_g3", "tiny_rnn", 3, 32, 10, "greedy", 3.0, True),
    ]
    only = [a for a in sys.argv[1:] if not a.startswith("-")]
    if only:  # regenerate just the named cases (the others stay byte-identical in git)
        cases = [c for c in cases if c[0] in only]
    for name, cfg, B, T, S, mode, gain, store_w in cases:
        c = tl.CONFIGS[cfg]
        dm = 0 if mode == "raw" else 1
        ref_las = tl.build_model(cfg, max_label_len=S, decode_mode=dm, seed=17, gain=gain, module=ref)
        our_las = tl.build_model(cfg, max_label_len=S, decode_mode=dm, seed=17, gain=gain, module=ours)
        sd_ref, sd_our = tl.state_dict_numpy(ref_las), tl.state_dict_numpy(our_las)
        assert list(sd_ref) == list(sd_our), "state_dict key order differs from the reference"
        for k in sd_ref:
            assert sd_ref[k].shape == sd_our[k].shape and np.array_equal(sd_ref[k], sd_our[k]), f"seeded init differs at {k}"
        our_las.load_state_dict(ref_las.state_dict(), strict=True)  # the drop-in contract

        x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
        gt = tl.onehot(labels, c["V"])
        out = {"x": x.numpy(), "labels": labels.numpy().astype(np.int32), "gain": gain, "seed": 17,
               "cfg": cfg, "mode": mode, "fingerprint": tl.weights_fingerprint(sd_ref)}
        for dt, tag in ((torch.float32, "f32"), (torch.float64, "f64")):
            enc, logp, attn = run_reference(ref_las, x, gt, mode == "tf", dt)
            out[f"enc_{tag}"], out[f"logp_{tag}"], out[f"attn_{tag}"] = enc, logp, attn
        d32 = np.abs(out["logp_f32"] - out["logp_f64"]).max()
        agree = (out["logp_f32"].argmax(-1) == out["logp_f64"].argmax(-1)).mean()
        tokens = len(np.unique(out["logp_f64"].argmax(-1)))
        if store_w:
            for k, v in sd_ref.items():
                out["w:" + k] = v
        else:
            out = compact(out)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(f"{name:18s} enc{out['enc_f32'].shape} logp{out['logp_f32'].shape} fp32-vs-fp64 logp {d32:.2e} "
              f"argmax agree {agree:.3f} distinct tokens {tokens} -> {os.path.getsize(path) / 1024:.0f} KiB")


if __name__ == "__main__":
    main()
