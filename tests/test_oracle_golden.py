"""Pins both CPU restatements (oracle/) against outputs of the reference itself (tests/golden/*.npz)."""
import glob

import numpy as np
import pytest
import torch

import las_testlib as tl
from oracle import las_oracle as O
from oracle.las_ref_torch import RefTorchLAS

CASES = tl.golden_cases()


def load_case(name):
    g = tl.load_golden(name)
    cfg = tl.CONFIGS[str(g["cfg"])]
    sd = {k[2:]: g[k] for k in g if k.startswith("w:")}
    if not sd:  # weights reproduced from the seed by our own parameter containers
        S = g["logp_f32"].shape[0]
        las = tl.build_model(str(g["cfg"]), max_label_len=S, seed=int(g["seed"]), gain=float(g["gain"]))
        sd = tl.state_dict_numpy(las)
        assert abs(tl.weights_fingerprint(sd) - float(g["fingerprint"])) < 1e-6 * abs(float(g["fingerprint"]))
    return g, cfg, sd


def test_golden_files_present():
    assert len(CASES) >= 10


@pytest.mark.parametrize("name", CASES)
def test_numpy_oracle_matches_reference(name):
    g, cfg, sd = load_case(name)
    mode = str(g["mode"])
    S = g["logp_f64"].shape[0]
    for dtype, tag, tol_enc, tol_lp in ((np.float64, "f64", 1e-12, 1e-11), (np.float32, "f32", 2e-6, 2e-5)):
        out = O.las_forward(g["x"], sd, cfg["L"], cfg["sl"], S, ground_truth=g["labels"] if mode == "tf" else None,
                            teacher_forced=(mode == "tf"), decode_mode=0 if mode == "raw" else 1, dtype=dtype)
        scale = 100.0 if float(g["gain"]) >= 6 and tag == "f32" else 1.0  # gain-6 is chaotic even fp32-vs-fp64
        if tag == "f32":  # no fp32 restatement can be closer to the reference's fp32 run than that run is to its own fp64 run
            scale = max(scale, 20.0 * float(np.abs(g["logp_f32"] - g["logp_f64"]).max()) / tol_lp)
        assert np.abs(out["enc"] - g[f"enc_{tag}"]).max() <= tol_enc * scale
        assert np.abs(out["logp"] - g[f"logp_{tag}"]).max() <= tol_lp * scale
        assert np.abs(out["attn"] - g[f"attn_{tag}"]).max() <= tol_lp * scale
        if tag == "f64":
            assert np.array_equal(out["tokens"], g["logp_f64"].argmax(-1))


@pytest.mark.parametrize("name", [c for c in CASES if not c.startswith(("paper", "tinymh", "tinynomlp", "tinygru", "tinyrnn"))])
def test_torch_restatement_matches_reference(name):
    """Same torch ops in the same order as the reference -> expected bit-identical on the same machine.  (The torch
    restatement is the timed CPU baseline of the benchmarked single-head LSTM configuration; the Attention / rnn_unit variants are
    covered by the numpy oracle above.)"""
    g, cfg, sd = load_case(name)
    mode = str(g["mode"])
    S = g["logp_f32"].shape[0]
    m = RefTorchLAS(sd, cfg["L"], cfg["sl"])
    gt = tl.onehot(torch.from_numpy(g["labels"]).long(), cfg["V"]) if mode == "tf" else None
    enc, logp, attn = m.forward(torch.from_numpy(g["x"]), S, gt, decode_mode=0 if mode == "raw" else 1)
    assert np.abs(enc.numpy() - g["enc_f32"]).max() <= 1e-6
    scale = 100.0 if float(g["gain"]) >= 6 else 1.0
    assert np.abs(logp.numpy() - g["logp_f32"]).max() <= 2e-6 * scale
    assert np.abs(attn.numpy() - g["attn_f32"]).max() <= 2e-6 * scale


def test_pyramid_fold_is_bit_exact_and_rejects_odd_lengths():
    x = np.arange(2 * 6 * 3, dtype=np.float32).reshape(2, 6, 3)
    y = O.pyramid_fold(x)
    assert y.shape == (2, 3, 6)
    assert np.array_equal(y[:, 1, :3], x[:, 2, :]) and np.array_equal(y[:, 1, 3:], x[:, 3, :])
    with pytest.raises(RuntimeError):
        O.pyramid_fold(np.zeros((2, 7, 3), np.float32))


def test_shard_invariance_of_oracle():
    """Utterances are independent (SURVEY.md 8e): full batch == concatenation of shards."""
    g, cfg, sd = load_case("tiny_tf_g3")
    full = O.las_forward(g["x"], sd, cfg["L"], cfg["sl"], 6, ground_truth=g["labels"], teacher_forced=True, dtype=np.float64)
    parts = [O.las_forward(g["x"][i:i + 1], sd, cfg["L"], cfg["sl"], 6, ground_truth=g["labels"][i:i + 1],
                           teacher_forced=True, dtype=np.float64) for i in range(g["x"].shape[0])]
    # BLAS picks different kernels for different batch sizes, so "bitwise" holds for torch (SURVEY.md 8e) but only
    # to rounding for numpy
    assert np.abs(full["logp"] - np.concatenate([p["logp"] for p in parts], axis=1)).max() < 1e-13


def test_solver_epilogue_restatement():
    rng = np.random.default_rng(0)
    logp = np.log(rng.dirichlet(np.ones(7), size=(2, 5)))  # [B,S,V]
    labels = np.array([[2, 3, 4, 1, 0], [5, 6, 1, 0, 0]])
    ref = torch.nn.NLLLoss(ignore_index=0)(torch.from_numpy(logp).permute(0, 2, 1), torch.from_numpy(labels))
    assert abs(O.nll_loss_ignore0(logp, labels) - float(ref)) < 1e-12
    assert O.letter_error_rate([[2, 3, 0, 4, 1, 5]], [[2, 3, 4, 1, 0, 0]]) == [0.0]
    assert O.letter_error_rate([[2, 2, 1]], [[2, 3, 4, 1]]) == [2 / 3]
    assert O.levenshtein("kitten", "sitting") == 3


def test_masked_listener_oracle_equals_torch_packed_sequence():
    """The length-mask extension's oracle is pinned to torch itself: per layer, pack_padded_sequence -> nn.LSTM ->
    pad_packed_sequence with lengths ceil-halved, which is what `listener_forward_masked` restates."""
    import torch
    from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

    torch.manual_seed(7)
    B, T, F, H, L = 5, 32, 40, 12, 3
    lstms = [torch.nn.LSTM((F if l == 0 else 2 * H) * 2, H, 1, bidirectional=True, batch_first=True).double() for l in range(L)]
    sd = {}
    for l, m in enumerate(lstms):
        for k, v in m.state_dict().items():
            sd[f"listener.pLSTM_layer{l}.BLSTM.{k}"] = v.numpy()
    x = torch.randn(B, T, F, dtype=torch.float64)
    lengths = torch.tensor([32, 27, 17, 8, 3])
    for b in range(B):
        x[b, lengths[b]:] = 0  # zero padding as utils/data.py:132
    out, lens = x, lengths.clone()
    with torch.no_grad():
        for m in lstms:
            xr = out.reshape(B, out.size(1) // 2, 2 * out.size(2))
            lens = (lens + 1) // 2
            packed = pack_padded_sequence(xr, lens, batch_first=True, enforce_sorted=False)
            out, _ = pad_packed_sequence(m(packed)[0], batch_first=True, total_length=xr.size(1))
    enc, enc_lens = O.listener_forward_masked(x.numpy(), lengths.numpy(), sd, L, dtype=np.float64)
    assert np.array_equal(enc_lens, lens.numpy())
    assert np.abs(enc - out.numpy()).max() < 1e-12
    # full lengths reproduce the unmasked (reference) listener exactly
    full, _ = O.listener_forward_masked(x.numpy(), np.full(B, T), sd, L, dtype=np.float64)
    assert np.abs(full - O.listener_forward(x.numpy(), sd, L, dtype=np.float64)).max() < 1e-13  # BLAS batch-size rounding only
