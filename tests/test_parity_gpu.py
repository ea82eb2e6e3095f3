"""GPU parity tests: the CUDA path (through the C ABI) vs the reference's frozen outputs and the numpy oracle.

Tolerances (BASELINE.json north_star): pyramid reshape / masks / argmax bit-exact; log-probs <= 1e-4 max-abs in
fp32 mode and <= 2e-2 in bf16 mode; greedy token sequences agree on >= 99% of characters.
"""
import glob
import os

import numpy as np
import pytest
import torch

import las_testlib as tl
from oracle import las_oracle as O

pytestmark = pytest.mark.gpu

CASES = tl.golden_cases()
# fp16 = the tensor-core kernels with IEEE fp16 operands (LAS_MODE_F16): 10 mantissa bits instead of bf16's 7, hence ~8x tighter bounds
TOL = {"fp32": dict(enc=2e-5, logp=1e-4, attn=2e-5), "bf16": dict(enc=3e-2, logp=2e-2, attn=1e-2),
       "fp16": dict(enc=4e-3, logp=3e-3, attn=1.5e-3)}


def precisions():
    from las_pytorch_b200 import _cabi

    out = ["fp32"]
    if _cabi.load_library().las_mode_available(_cabi.MODE_BF16):
        out.append("bf16")
    if _cabi.load_library().las_mode_available(_cabi.MODE_F16):
        out.append("fp16")
    return out


def load_case(name, precision):
    g = tl.load_golden(name)
    cfg = str(g["cfg"])
    mode = str(g["mode"])
    S = g["logp_f64"].shape[0]
    las = tl.build_model(cfg, max_label_len=S, decode_mode=0 if mode == "raw" else 1, seed=int(g["seed"]),
                         gain=float(g["gain"]), precision=precision)
    sd = {k[2:]: torch.from_numpy(g[k]) for k in g if k.startswith("w:")}
    if sd:
        las.load_state_dict(sd, strict=True)
    else:
        fp = tl.weights_fingerprint(tl.state_dict_numpy(las))
        assert abs(fp - float(g["fingerprint"])) < 1e-6 * abs(float(g["fingerprint"]))
    return g, tl.CONFIGS[cfg], las.cuda(), mode


def run_ours(las, x, labels, V, mode):
    x = x.cuda()
    gt = tl.onehot(labels, V).cuda() if mode == "tf" else None
    np.random.seed(0)
    preds, attns = las(x, gt, 1.1 if mode == "tf" else 0.0, is_training=(mode == "tf"))
    enc = las.listener(x)
    torch.cuda.synchronize()
    if len(attns[0]) == 1:
        attn = torch.stack([a[0] for a in attns])
    else:  # multi_head > 1: one [B,U] tensor per head and step (model/las_model.py:299) -> [S,heads,B,U]
        attn = torch.stack([torch.stack(list(a)) for a in attns])
    return enc.cpu().numpy(), torch.stack(preds).cpu().numpy(), attn.cpu().numpy()


@pytest.mark.parametrize("precision", precisions())
@pytest.mark.parametrize("name", CASES)
def test_matches_reference_golden(name, precision):
    # (row f4 variants -- multi-head, no-MLP attention, GRU / RNN cells -- run in the bf16 mode through the generic tensor-core path)
    g, cfg, las, mode = load_case(name, precision)
    tol = TOL[precision]
    enc, logp, attn = run_ours(las, torch.from_numpy(g["x"]), torch.from_numpy(g["labels"]).long(), cfg["V"], mode)
    # the reference's own fp32-vs-fp64 gap bounds what any fp32 implementation can promise (gain-6 is chaotic)
    ref_noise = float(np.abs(g["logp_f32"] - g["logp_f64"]).max())
    slack = max(1.0, 20.0 * ref_noise / tol["logp"])
    chaotic_bf16 = precision != "fp32" and float(g["gain"]) >= 6
    if chaotic_bf16:
        # gain-6 weights are chaotic (SURVEY.md A.6: the reference's own fp32 run is 5e-4 away from its fp64 run, 28x its usual
        # noise).  bf16 operand rounding (listener error 7e-2 here) flips the peaked attention onto other frames, so only
        # the listener is held to a (5x) bound in this regime; measured log-prob error is recorded in profiles/ and DESIGN.md.
        slack = 5.0
    sens = dict(enc=0.0, logp=0.0, attn=0.0)
    if precision != "fp32" and cfg.get("unit", "LSTM") != "LSTM":
        # Ungated tanh / GRU recurrences at gain 3 amplify operand rounding far more than the LSTM does: the ORACLE itself, fed
        # bf16-rounded inputs and 2-D weights (fp64 arithmetic), moves the tiny GRU / RNN goldens by 4e-2 / 5e-2 in the listener and
        # up to 0.6 in the log-probs.  Calibrate on the spot: the bound is 3x that sensitivity where it exceeds the mode's tolerance.
        def bf(a):
            return torch.from_numpy(np.asarray(a, np.float32)).to(torch.bfloat16 if precision == "bf16" else torch.float16).float().numpy()

        sd_full = tl.state_dict_numpy(las)
        sd_b = {k: (bf(v) if v.ndim == 2 else v) for k, v in sd_full.items()}
        rb = O.las_forward(bf(g["x"]), sd_b, cfg["L"], cfg["sl"], logp.shape[0], ground_truth=g["labels"], teacher_forced=True, dtype=np.float64)
        sens = dict(enc=float(np.abs(rb["enc"] - g["enc_f64"]).max()), logp=float(np.abs(rb["logp"] - g["logp_f64"]).max()),
                    attn=float(np.abs(rb["attn"] - g["attn_f64"]).max()))
    tol = {k: max(tol[k], 3.0 * sens[k]) for k in tol}
    assert enc.shape == g["enc_f64"].shape and logp.shape == g["logp_f64"].shape and attn.shape == g["attn_f64"].shape
    if mode == "tf" or precision == "fp32":
        assert np.abs(enc - g["enc_f64"]).max() <= tol["enc"] * slack
        if not chaotic_bf16:
            assert np.abs(logp - g["logp_f64"]).max() <= tol["logp"] * slack
            assert np.abs(attn - g["attn_f64"]).max() <= tol["attn"] * slack
    ref_tok = g["logp_f64"].argmax(-1)
    srt = np.sort(g["logp_f64"], axis=-1)
    margin = srt[..., -1] - srt[..., -2]
    tok = logp.argmax(-1)
    if mode == "tf" and not chaotic_bf16:
        # argmax bit-exact wherever the oracle's top-2 margin exceeds twice the log-prob tolerance (two log-probs can each move by
        # the tolerance); the mask is proportional to the tolerance, and must keep a stated share of the positions
        safe = margin > 2 * tol["logp"] * slack
        if precision == "fp32":
            assert safe.mean() >= 0.9, safe.mean()  # (bf16: the default-init goldens have margins of ~4e-3, far below 4e-2; the
            # share kept at the benchmarked shapes is asserted in tests/test_benchmark_shapes_gpu.py)
        assert np.array_equal(tok[safe], ref_tok[safe])
    elif precision == "fp32":
        assert (tok == ref_tok).mean() >= 0.99
    elif mode == "greedy":
        # bf16, free running: whatever trajectory the decoder follows, each step's log-probs must be the oracle's for the tokens that
        # were fed back (teacher-forced re-scoring of our own output)
        rescored = O.las_forward(g["x"], tl.state_dict_numpy(las), cfg["L"], cfg["sl"], logp.shape[0], ground_truth=tok.T,
                                 teacher_forced=True, dtype=np.float64)
        assert np.abs(logp - rescored["logp"]).max() <= tol["logp"] * slack
    assert np.abs(np.exp(logp).sum(-1) - 1).max() < 1e-4
    assert np.abs(attn.sum(-1) - 1).max() < 1e-4


@pytest.mark.parametrize("precision", precisions())
def test_against_numpy_oracle_on_seeded_inputs(precision):
    """Same seeded inputs/weights through the CUDA path and the fp64 numpy oracle (sizes the oracle does in seconds)."""
    cfgname, B, T, S = "small", 6, 256, 40
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=23, gain=3.0, precision=precision)
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=23, pad_tail=32)
    ref_tf = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, ground_truth=labels.numpy(), teacher_forced=True, dtype=np.float64)
    ref_gr = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, dtype=np.float64)
    las = las.cuda()
    tol = TOL[precision]
    enc, logp, attn = run_ours(las, x, labels, c["V"], "tf")
    assert np.abs(enc - ref_tf["enc"]).max() <= tol["enc"]
    assert np.abs(logp - ref_tf["logp"]).max() <= tol["logp"]
    assert np.abs(attn - ref_tf["attn"]).max() <= tol["attn"]
    _, logp_g, _ = run_ours(las, x, labels, c["V"], "greedy")
    agree = (logp_g.argmax(-1) == ref_gr["tokens"]).mean()
    floor = 0.99
    if precision != "fp32":
        # bf16 GEMM operands move log-probs by ~4e-3, enough to flip a near-tie and send a free-running utterance down another
        # trajectory.  Calibrate on the spot: the ORACLE with nothing but its 2-D weights rounded to bf16 vs itself (see
        # tests/test_benchmark_shapes_gpu.py); ours must be no worse than that minus 0.05.
        rdt = torch.bfloat16 if precision == "bf16" else torch.float16
        sd_b = {k: (torch.from_numpy(v).to(rdt).float().numpy() if v.ndim == 2 else v) for k, v in sd.items()}
        ref_b = O.las_forward(x.numpy(), sd_b, c["L"], c["sl"], S, dtype=np.float64)
        floor = min(0.99, float((ref_b["tokens"] == ref_gr["tokens"]).mean()) - 0.05)
        tok = logp_g.argmax(-1)
        rescored = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, ground_truth=tok.T, teacher_forced=True, dtype=np.float64)
        assert np.abs(logp_g - rescored["logp"]).max() <= tol["logp"]  # every step of the trajectory we followed is right
    assert agree >= floor, f"greedy agreement {agree:.3f} < {floor:.3f}"
    if precision == "fp32":
        assert np.abs(logp_g - ref_gr["logp"]).max() <= tol["logp"]
        assert np.array_equal(las.speller.last_tokens.cpu().numpy(), logp_g.argmax(-1))


@pytest.mark.parametrize("precision", precisions())
def test_full_size_properties(precision):
    """BASELINE.json config 3 shape (paper LAS, batch 64 x 1600 frames) through size-independent properties:
    normalisation, determinism, and shard invariance (an utterance's result does not depend on its batch)."""
    c = tl.CONFIGS["paper"]
    B, T, S = 64, 1600, 24
    las = tl.build_model("paper", max_label_len=S, seed=17, gain=3.0, precision=precision).cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17)
    x = x.cuda()
    enc = las.listener(x)
    assert enc.shape == (B, T // 8, 2 * c["H"])
    assert torch.isfinite(enc).all() and float(enc.abs().max()) <= 1.0  # h = o * tanh(c) is bounded by 1
    preds, attns = las(x, None, 0.0, is_training=False)
    logp = torch.stack(preds)
    attn = torch.stack([a[0] for a in attns])
    assert logp.shape == (S, B, c["V"]) and attn.shape == (S, B, T // 8)
    assert float((logp.exp().sum(-1) - 1).abs().max()) < 1e-4
    assert float((attn.sum(-1) - 1).abs().max()) < 1e-4
    # determinism
    preds2, _ = las(x, None, 0.0, is_training=False)
    assert torch.equal(torch.stack(preds2), logp)
    # shard invariance: two half batches == the full batch (what sharding over GPUs relies on, SURVEY.md 8e)
    halves = [las(x[i:i + B // 2], None, 0.0, is_training=False)[0] for i in (0, B // 2)]
    sharded = torch.cat([torch.stack(h) for h in halves], dim=1)
    assert torch.equal(sharded, logp)  # both modes: every kernel variant a batch size can select accumulates in the same order


@pytest.mark.parametrize("name", ["paper_greedy_g3", "small_greedy_g3"])
def test_bf16_greedy_agreement_on_named_shapes(name):
    """north_star: free-running greedy token sequences agree with the reference on >= 99 % of characters, also in the
    bf16-GEMM mode, at the shapes the benchmark names (paper / small LAS)."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    g, cfg, las, mode = load_case(name, "bf16")
    _, logp, _ = run_ours(las, torch.from_numpy(g["x"]), torch.from_numpy(g["labels"]).long(), cfg["V"], mode)
    agree = (logp.argmax(-1) == g["logp_f64"].argmax(-1)).mean()
    assert agree >= 0.99, f"greedy agreement {agree:.4f}"


@pytest.mark.parametrize("precision", precisions())
@pytest.mark.parametrize("cfgname", ["small", "odd"])
def test_index_teacher_forcing_equals_onehot(cfgname, precision):
    """Row f2 extension: [B,S] label indices feed the same decoder as the reference's one-hot tensor.  In bf16 mode the index
    path adds the word column of W_ih in the LSTM epilogue instead of multiplying a one-hot atom on the tensor core."""
    c = tl.CONFIGS[cfgname]
    B, T, S = 5, 64, 12
    las = tl.build_model(cfgname, max_label_len=S, seed=29, gain=3.0, precision=precision)
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=29)
    ref = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, ground_truth=labels.numpy(), teacher_forced=True, dtype=np.float64)
    las = las.cuda()
    np.random.seed(0)
    p_idx, _ = las(x.cuda(), labels.cuda(), 1.1, is_training=True)
    np.random.seed(0)
    p_hot, _ = las(x.cuda(), tl.onehot(labels, c["V"]).cuda(), 1.1, is_training=True)
    p_idx, p_hot = torch.stack(p_idx).cpu().numpy(), torch.stack(p_hot).cpu().numpy()
    tol = TOL[precision]["logp"]
    assert np.abs(p_idx - ref["logp"]).max() <= tol and np.abs(p_hot - ref["logp"]).max() <= tol
    assert np.abs(p_idx - p_hot).max() <= (1e-5 if precision == "fp32" else 2e-3)  # same numbers up to fp32 summation order


def test_bf16_forward_step_state_roundtrip():
    """Speller.forward_step in bf16 mode: state / word / context handed in and out step by step equals one fused decode."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS["small"]
    S = 4
    las = tl.build_model("small", max_label_len=S, seed=31, gain=3.0, precision="bf16")
    sd = tl.state_dict_numpy(las)
    las = las.cuda()
    enc = torch.tanh(torch.randn(3, 16, 2 * c["H"], generator=torch.Generator().manual_seed(4)))
    ref = O.speller_forward(enc.numpy(), sd, c["sl"], S, dtype=np.float64)
    encd = enc.cuda()
    fused, _ = las.speller(encd, None, 0.0)
    word = torch.zeros(3, 1, c["V"], device="cuda")
    word[:, :, 0] = 1
    rnn_in = torch.cat([word, encd[:, 0:1, :]], dim=-1)
    hidden = None
    for s in range(S):
        raw_pred, hidden, context, score = las.speller.forward_step(rnn_in, hidden, encd)
        assert np.abs(raw_pred.cpu().numpy() - ref["logp"][s]).max() <= 2e-2
        assert float((raw_pred - fused[s]).abs().max()) <= 5e-3  # the state leaves / re-enters through fp32 and bf16 copies
        nxt = torch.nn.functional.one_hot(raw_pred.argmax(-1), c["V"]).float().unsqueeze(1)
        rnn_in = torch.cat([nxt, context.unsqueeze(1)], dim=-1)


def test_bf16_length_mask():
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS["small"]
    las = tl.build_model("small", max_label_len=6, seed=3, gain=3.0, precision="bf16")
    sd = tl.state_dict_numpy(las)
    las = las.cuda()
    enc = torch.tanh(torch.randn(4, 24, 2 * c["H"], generator=torch.Generator().manual_seed(2)))
    lens = torch.tensor([24, 17, 5, 1])
    ref = O.speller_forward(enc.numpy(), sd, c["sl"], 6, dtype=np.float64, enc_lengths=lens.numpy())
    preds, attns = las.speller(enc.cuda(), None, 0.0, enc_lengths=lens)
    attn = torch.stack([a[0] for a in attns]).cpu().numpy()
    assert np.abs(torch.stack(preds).cpu().numpy() - ref["logp"]).max() <= 2e-2
    assert np.array_equal(attn[:, 2, 5:], np.zeros_like(attn[:, 2, 5:]))  # masked steps get exactly zero weight
    assert np.abs(attn.sum(-1) - 1).max() < 1e-4


@pytest.mark.parametrize("precision", precisions())
@pytest.mark.parametrize("cfgname", ["small", "odd"])
def test_listener_length_masks(cfgname, precision):
    """Length-mask extension (north_star): BLSTMs and attention skip the padding; the oracle is pinned to torch's
    packed-sequence LSTM on CPU.  An utterance's result no longer depends on how much padding follows it."""
    c = tl.CONFIGS[cfgname]
    B, T, S = 6, 64, 6
    las = tl.build_model(cfgname, max_label_len=S, seed=41, gain=3.0, precision=precision)
    sd = tl.state_dict_numpy(las)
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=41)
    lengths = torch.tensor([64, 57, 40, 33, 9, 2])
    for b in range(B):
        x[b, lengths[b]:] = 0
    ref_enc, ref_lens = O.listener_forward_masked(x.numpy(), lengths.numpy(), sd, c["L"], dtype=np.float64)
    ref = O.speller_forward(ref_enc, sd, c["sl"], S, dtype=np.float64, enc_lengths=ref_lens)
    las = las.cuda()
    enc, enc_lens = las.listener(x.cuda(), input_lengths=lengths)
    tol = TOL[precision]
    assert np.array_equal(enc_lens.cpu().numpy(), ref_lens)  # mask indices bit-exact
    assert np.abs(enc.cpu().numpy() - ref_enc).max() <= tol["enc"]
    for b in range(B):  # outputs past the valid length are exactly zero
        assert float(enc[b, int(ref_lens[b]):].abs().max() if int(ref_lens[b]) < enc.size(1) else 0.0) == 0.0
    preds, attns = las(x.cuda(), None, 0.0, is_training=False, input_lengths=lengths)
    logp = torch.stack(preds).cpu().numpy()
    if precision == "fp32":
        assert np.abs(logp - ref["logp"]).max() <= tol["logp"]
    # free running under operand rounding: the oracle re-scores the trajectory that was actually followed (a near-tie may flip a token)
    ref_rs = O.speller_forward(ref_enc, sd, c["sl"], S, ground_truth=logp.argmax(-1).T, dtype=np.float64, enc_lengths=ref_lens)
    assert np.abs(logp - ref_rs["logp"]).max() <= tol["logp"]
    # padding invariance: the same utterances with 32 more padded frames give the same valid outputs
    xp = torch.cat([x, torch.zeros(B, 32, c["F"])], dim=1)
    enc2, enc_lens2 = las.listener(xp.cuda(), input_lengths=lengths)
    assert torch.equal(enc_lens2, enc_lens)
    assert torch.equal(enc2[:, : enc.size(1)], enc) and float(enc2[:, enc.size(1):].abs().max()) == 0.0
    # lengths == T reproduce the reference (unmasked) path bit for bit
    enc_full, _ = las.listener(x.cuda(), input_lengths=torch.full((B,), T))
    assert torch.equal(enc_full, las.listener(x.cuda()))


def test_bf16_listener_overlap_is_bit_identical_to_sequential():
    """The input-projection GEMM running next to the recurrence (tile flags + watcher warp) must give exactly what the
    GEMM-then-recurrence order gives: same arithmetic, only the schedule differs."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS["paper"]
    lis = tl.build_model("paper", max_label_len=4, seed=47, gain=3.0, precision="bf16").listener.cuda()
    x, _ = tl.make_inputs(24, 512, c["F"], 4, c["V"], seed=47)
    x = x.cuda()
    try:
        lib.las_debug_set_option(6, 0)
        seq = lis(x).clone()
        lib.las_debug_set_option(6, 1)
        outs = [lis(x).clone() for _ in range(3)]
    finally:
        lib.las_debug_set_option(6, 1)
    for o in outs:
        assert torch.equal(o, seq)


def test_bf16_decoder_single_3d_copy_matches_per_atom_copies():
    """The decoder's activation parts arrive as ONE 3-D TMA copy when Hs and E are multiples of 64, and as one 2-D copy per
    64-column atom otherwise (las_debug_set_option(5, 4) forces the latter): same bytes in shared memory, so greedy tokens,
    log-probs and attention must be bit-identical."""
    if "bf16" not in precisions():
        pytest.skip("bf16 path not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS["paper"]
    S = 24
    las = tl.build_model("paper", max_label_len=S, seed=61, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(10, 256, c["F"], S, c["V"], seed=61)
    enc = las.listener(x.cuda())

    def run():
        pred, att = las.speller(enc, None, 0.0)
        return torch.stack(pred).clone(), torch.stack([a[0] for a in att]).clone()

    try:
        lib.las_debug_set_option(5, 4)
        p2, a2 = run()
    finally:
        lib.las_debug_set_option(5, 0)
    p3, a3 = run()
    assert torch.equal(p2, p3) and torch.equal(a2, a3)
    assert torch.isfinite(p3).all()


def test_bf16_long_encoder_context_paths():
    """Long encoders (BASELINE config 4: 3000 frames -> U = 375): enc[b]^T no longer fits ONE attention CTA's tensor memory.
    Default: a cluster of two CTAs attends each utterance, each with half of the encoder steps fully in tensor memory, partial
    softmax / context combined through DSMEM (las_debug_set_option(11, 1)).  Alternatives kept for A/B and for shapes the split does
    not cover: hybrid (two of the four 128-feature tiles on the UMMA, two on the CUDA cores; option 11 = 0) and CUDA cores only
    (option 2 = 0).  All three against the fp64 oracle -- teacher forced, with a length mask that leaves the second CTA of some
    pairs nothing to attend, and free running -- and against each other."""
    if "bf16" not in precisions():
        pytest.skip("bf16 path not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS["paper"]
    B, T, S = 5, 3000, 12
    las = tl.build_model("paper", max_label_len=S, seed=71, gain=3.0, precision="bf16")
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=71)
    ref = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, ground_truth=labels.numpy(), teacher_forced=True, dtype=np.float64)
    las = las.cuda()
    out = {}
    variants = {"split": (11, 1, 2, 1), "hybrid": (11, 0, 2, 1), "cuda_cores": (11, 0, 2, 0)}
    for name, (k1, v1, k2, v2) in variants.items():
        try:
            lib.las_debug_set_option(k1, v1)
            lib.las_debug_set_option(k2, v2)
            out[name] = run_ours(las, x, labels, c["V"], "tf")
        finally:
            lib.las_debug_set_option(11, 1)
            lib.las_debug_set_option(2, 1)
    for name in variants:
        _, logp, attn = out[name]
        assert np.abs(logp - ref["logp"]).max() <= TOL["bf16"]["logp"], name
        assert np.abs(attn - ref["attn"]).max() <= TOL["bf16"]["attn"], name
        assert np.abs(attn.sum(-1) - 1).max() < 1e-4, name
    assert np.abs(out["cuda_cores"][1] - out["hybrid"][1]).max() <= 5e-3  # the context paths differ only by the bf16 rounding of the scores
    assert np.abs(out["split"][1] - out["hybrid"][1]).max() <= 5e-3
    assert not np.array_equal(out["cuda_cores"][1], out["hybrid"][1]) and not np.array_equal(out["split"][1], out["hybrid"][1])
    # length masks: utterance 1 ends inside the first CTA's half (the second CTA's partial sums are all zero), utterance 2 inside the second's
    enc = las.listener(x.cuda())
    lens = torch.tensor([375, 100, 250, 192, 193], dtype=torch.int32)
    ref_m = O.speller_forward(ref["enc"], sd, c["sl"], S, labels.numpy(), 1, np.float64, enc_lengths=lens.numpy())
    np.random.seed(0)
    preds, attns = las.speller(enc, labels.cuda(), 1.1, enc_lengths=lens.cuda())
    attn_m = torch.stack([a[0] for a in attns]).cpu().numpy()
    for b_, n in enumerate(lens.tolist()):
        assert float(np.abs(attn_m[:, b_, n:]).max() if n < 375 else 0.0) == 0.0       # nothing attended past the length
        assert np.abs(attn_m[:, b_, :n].sum(-1) - 1).max() < 1e-4
    assert np.abs(torch.stack(preds).cpu().numpy() - ref_m["logp"]).max() <= TOL["bf16"]["logp"]
    assert np.abs(attn_m - ref_m["attn"]).max() <= TOL["bf16"]["attn"]
    _, logp_g, _ = run_ours(las, x, labels, c["V"], "greedy")
    assert np.isfinite(logp_g).all() and np.abs(np.exp(logp_g).sum(-1) - 1).max() < 1e-4


@pytest.mark.parametrize("precision", precisions())
def test_edge_shapes_single_utterance_single_step_single_encoder_frame(precision):
    """Smallest shapes the path accepts: one utterance, T = 2^L (one encoder step: the softmax is over a single frame),
    one decode step; and a ragged batch (B = 3) that fills neither a 16-utterance recurrence chunk nor a TMEM quadrant."""
    c = tl.CONFIGS["small"]
    for B, T, S in ((1, 4, 1), (1, 8, 3), (3, 12, 2)):
        las = tl.build_model("small", max_label_len=S, seed=53, gain=3.0, precision=precision)
        sd = tl.state_dict_numpy(las)
        x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=53)
        ref = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, dtype=np.float64)
        las = las.cuda()
        preds, attns = las(x.cuda(), None, 0.0, is_training=False)
        logp = torch.stack(preds).cpu().numpy()
        attn = torch.stack([a[0] for a in attns]).cpu().numpy()
        assert logp.shape == (S, B, c["V"]) and attn.shape == (S, B, T // 4)
        assert np.abs(logp - ref["logp"]).max() <= TOL[precision]["logp"]
        assert np.abs(attn.sum(-1) - 1).max() < 1e-5
        if T // 4 == 1:
            assert np.array_equal(attn, np.ones_like(attn))  # a single encoder frame gets all the weight, exactly


def test_error_paths_raise_instead_of_falling_back():
    """No CPU fallback and no silent substitution: every unsupported request raises with a message that says what to do."""
    import las_pytorch_b200 as ours
    from las_pytorch_b200 import _cabi

    las = tl.build_model("tiny", max_label_len=3, seed=1, gain=1.0)
    x = torch.randn(2, 16, 40)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        las.listener(x)  # CPU tensor
    las = las.cuda()
    with pytest.raises(RuntimeError):  # T not divisible by 2^L: the reference's view() raises too (model/las_model.py:87)
        las.listener(torch.randn(2, 18, 40, device="cuda"))
    with pytest.raises(RuntimeError, match="feature dim"):
        las.listener(torch.randn(2, 16, 39, device="cuda"))
    with pytest.raises(ValueError, match="2\\*listener_hidden_size"):  # Hs != 2H cannot work in the reference either (SURVEY A.4)
        ours.Speller(30, 48, "LSTM", 2, 5, True, 16, "relu", 16, 1, 1)
    with pytest.raises(NotImplementedError):
        ours.Listener(40, 16, 2, "QRNN")  # only what getattr(nn, ...) would give the reference: LSTM, GRU, RNN
    with pytest.raises(ValueError):
        ours.Speller(30, 32, "LSTM", 2, 5, True, 16, "relu", 16, 1, 3)  # decode_mode is 0, 1 or 2 in the reference
    if "bf16" in precisions():
        # shapes outside the persistent decoder (here V > 64, its word atom) run on the generic tensor-core path instead of raising
        big_v = ours.Speller(80, 32, "LSTM", 2, 3, True, 16, "relu", 16, 1, 1, precision="bf16").cuda()
        preds, _ = big_v(torch.randn(2, 4, 32, device="cuda"), None, 0.0)
        assert len(preds) == 3 and preds[0].shape == (2, 80) and float((torch.stack(preds).exp().sum(-1) - 1).abs().max()) < 1e-4
    # the library reports a bad status instead of aborting
    lib = _cabi.load_library()
    d = _cabi.ListenerDims(2, 15, 40, 16, 2)
    import ctypes as C
    assert lib.las_listener_forward(None, None, C.byref(d), 0, None, None, 0, None) != 0
    assert b"" != lib.las_last_error()


@pytest.mark.parametrize("precision", precisions())
def test_decode_mode_2_sampling(precision):
    """decode_mode 2 (model/las_model.py:229-234): the fed-back word is a draw from Categorical(probs = log-probs), i.e.
    p_i = logp_i / sum_j logp_j (SURVEY.md A.5.6).  The draws cannot equal torch's generator stream, so the check is:
    (1) re-scoring the sampled tokens through the oracle in teacher-forced mode reproduces every log-prob (the sampled word really
    is what was fed back); (2) runs are reproducible under torch.manual_seed and differ across seeds; (3) first-step draws over
    many identical utterances follow the reference's (inverted) distribution."""
    c = tl.CONFIGS["small"]
    B, T, S = 6, 64, 10
    las = tl.build_model("small", max_label_len=S, decode_mode=2, seed=59, gain=3.0, precision=precision)
    sd = tl.state_dict_numpy(las)
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=59)
    las = las.cuda()
    torch.manual_seed(1234)
    preds, _ = las(x.cuda(), None, 0.0, is_training=False)
    toks = las.speller.last_tokens.cpu().numpy().T  # [B,S] sampled tokens
    ref = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, ground_truth=toks, teacher_forced=True, dtype=np.float64)
    assert np.abs(torch.stack(preds).cpu().numpy() - ref["logp"]).max() <= TOL[precision]["logp"]
    assert not np.array_equal(toks, ref["tokens"].T)  # sampling from the inverted distribution is not the argmax path
    torch.manual_seed(1234)
    las(x.cuda(), None, 0.0, is_training=False)
    assert np.array_equal(las.speller.last_tokens.cpu().numpy().T, toks)
    torch.manual_seed(4321)
    las(x.cuda(), None, 0.0, is_training=False)
    assert not np.array_equal(las.speller.last_tokens.cpu().numpy().T, toks)
    # distribution of the first draw: 64 copies of one utterance x 40 seeds = 2560 draws
    xr = x[:1].repeat(64, 1, 1).cuda()
    counts = np.zeros(c["V"])
    for seed in range(40):
        torch.manual_seed(seed)
        las(xr, None, 0.0, is_training=False)
        counts += np.bincount(las.speller.last_tokens[0].cpu().numpy(), minlength=c["V"])
    lp0 = ref["logp"][0, 0]
    p = lp0 / lp0.sum()
    n = counts.sum()
    z = (counts - n * p) / np.sqrt(n * p * (1 - p))
    assert np.abs(z).max() < 5.0, (counts, n * p)


@pytest.mark.parametrize("precision", precisions())
def test_single_layer_speller_and_padded_index_targets(precision):
    """A one-layer speller (the same LSTM CTA is both the layer that takes [word | context] and the one that feeds the attention)
    and index targets with padding: index -1 feeds the zero vector, exactly like an all-zero row of the reference's one-hot tensor
    (what collate_fn pads with, utils/data.py:133-136)."""
    cfg = dict(F=40, H=32, L=2, sl=1, V=30, D=16)
    B, T, S = 5, 32, 7
    las = tl.build_model(cfg, max_label_len=S, seed=61, gain=3.0, precision=precision)
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, cfg["F"], S, cfg["V"], seed=61)
    dense = tl.onehot(labels, cfg["V"]).clone()
    padded = labels.clone()
    dense[:, -2:, :] = 0   # padded steps: all-zero rows
    padded[:, -2:] = -1
    ref = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, ground_truth=dense.numpy().astype(np.float64), teacher_forced=True, dtype=np.float64)
    las = las.cuda()
    tol = TOL[precision]["logp"]
    for gt in (dense.cuda(), padded.cuda()):
        np.random.seed(0)
        preds, _ = las(x.cuda(), gt, 1.1, is_training=True)
        assert np.abs(torch.stack(preds).cpu().numpy() - ref["logp"]).max() <= tol
    greedy_ref = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, dtype=np.float64)
    preds, _ = las(x.cuda(), None, 0.0, is_training=False)
    lg = torch.stack(preds).cpu().numpy()
    if precision == "fp32":
        assert np.abs(lg - greedy_ref["logp"]).max() <= tol
    else:
        # a 32-unit net flips near-tied tokens under bf16 rounding and then follows another trajectory; what must hold is that every
        # step's log-probs are the oracle's for the tokens that were actually fed back
        toks = las.speller.last_tokens.cpu().numpy().T
        rescored = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, ground_truth=toks, teacher_forced=True, dtype=np.float64)
        assert np.abs(lg - rescored["logp"]).max() <= tol


def test_two_devices_from_two_host_threads():
    """The boundary's threading contract (SURVEY.md 8b: nn.DataParallel runs forward on one thread per GPU replica, train.py:76-78):
    two host threads drive two devices concurrently through the same library and each gets what a lone run gets."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import copy
    import threading

    c = tl.CONFIGS["small"]
    B, T, S = 8, 128, 12
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=67)
    for precision in precisions():
        base = tl.build_model("small", max_label_len=S, seed=67, gain=3.0, precision=precision)
        lone = torch.stack(copy.deepcopy(base).cuda(0)(x.cuda(0), None, 0.0, is_training=False)[0]).cpu()
        out, err = {}, []

        def work(dev):
            try:
                with torch.cuda.device(dev):
                    m = copy.deepcopy(base).cuda(dev)
                    for _ in range(3):
                        r = torch.stack(m(x.cuda(dev), None, 0.0, is_training=False)[0])
                    out[dev] = r.cpu()
            except Exception as e:  # noqa: BLE001
                err.append(e)

        ts = [threading.Thread(target=work, args=(d,)) for d in (0, 1)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert not err, err
        assert torch.equal(out[0], lone) and torch.equal(out[1], lone)


def test_shipped_config_size_decodes_in_both_modes():
    """config/librispeech-config.yaml:13-34 ships listener 512x3 / speller 1024x2.  The fp32 path takes any size; the bf16 listener
    takes H = 512 (16-CTA clusters); 1024-wide decoder cells (34 MB of LSTM weights) exceed what the persistent decoder keeps on
    chip, so the bf16 mode decodes them on the generic tensor-core path (weights streamed through a tcgen05 GEMM per cell and
    step) -- within the bf16 tolerance of the oracle, teacher-forced and re-scored free-running."""
    cfg = dict(F=40, H=512, L=3, sl=2, V=30, D=64)
    B, T, S = 3, 64, 6
    las = tl.build_model(cfg, max_label_len=S, seed=71, gain=2.0, precision="fp32")
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, cfg["F"], S, cfg["V"], seed=71)
    ref = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, dtype=np.float64)
    ref_tf = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, ground_truth=labels.numpy(), teacher_forced=True, dtype=np.float64)
    las = las.cuda()
    preds, _ = las(x.cuda(), None, 0.0, is_training=False)
    assert np.abs(torch.stack(preds).cpu().numpy() - ref["logp"]).max() <= 1e-4
    if "bf16" in precisions():
        lasb = tl.build_model(cfg, max_label_len=S, seed=71, gain=2.0, precision="bf16").cuda()
        enc = lasb.listener(x.cuda())  # H = 512 is within the bf16 listener's range
        assert np.abs(enc.cpu().numpy() - ref["enc"]).max() <= 3e-2
        np.random.seed(0)
        preds, attns = lasb(x.cuda(), labels.cuda(), 1.1, is_training=True)
        assert np.abs(torch.stack(preds).cpu().numpy() - ref_tf["logp"]).max() <= 2e-2
        assert np.abs(torch.stack([a[0] for a in attns]).cpu().numpy() - ref_tf["attn"]).max() <= 1e-2
        preds, _ = lasb(x.cuda(), None, 0.0, is_training=False)
        logp = torch.stack(preds).cpu().numpy()
        rescored = O.las_forward(x.numpy(), sd, cfg["L"], cfg["sl"], S, ground_truth=logp.argmax(-1).T, teacher_forced=True, dtype=np.float64)
        assert np.abs(logp - rescored["logp"]).max() <= 2e-2
        # forward_step / state hand-over and the <eos> early exit contract work on this path too
        lasb.speller.eos_token, lasb.speller.early_exit_every = int(logp.argmax(-1)[0, 0]), 2
        lasb.speller(enc[:1], None, 0.0, early_exit=True)
        assert int(lasb.speller.last_steps_done) == 2


def test_bf16_batch_larger_than_one_decoder_launch():
    """The persistent decoder covers at most 64 utterances per launch (one attention CTA each); larger batches are decoded
    in chunks.  70 utterances must equal the same utterances decoded as 64 + 6."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS["small"]
    B, T, S = 70, 64, 8
    las = tl.build_model("small", max_label_len=S, seed=43, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=43)
    x = x.cuda()
    full = torch.stack(las(x, None, 0.0, is_training=False)[0])
    tok_full = las.speller.last_tokens.clone()
    a = torch.stack(las(x[:64], None, 0.0, is_training=False)[0])
    b = torch.stack(las(x[64:], None, 0.0, is_training=False)[0])
    both = torch.cat([a, b], dim=1)
    assert full.shape == (S, B, c["V"]) and tok_full.shape == (S, B)
    assert torch.equal(full, both)  # launch groups of 64 + 6 utterances vs one call: bit-identical
    assert float((full.exp().sum(-1) - 1).abs().max()) < 1e-4


def test_forward_step_and_attention_api():
    """Speller.forward_step / Attention.forward (model/las_model.py:178-184, 275-297) against the oracle."""
    c = tl.CONFIGS["tiny"]
    las = tl.build_model("tiny", max_label_len=5, seed=3, gain=3.0)
    sd = tl.state_dict_numpy(las)
    las = las.cuda()
    g = torch.Generator().manual_seed(1)
    enc = torch.tanh(torch.randn(3, 8, 2 * c["H"], generator=g))
    ref = O.speller_forward(enc.numpy(), sd, c["sl"], 3, dtype=np.float64)
    encd = enc.cuda()
    word = torch.zeros(3, 1, c["V"], device="cuda")
    word[:, :, 0] = 1
    rnn_in = torch.cat([word, encd[:, 0:1, :]], dim=-1)
    hidden = None
    for s in range(3):
        raw_pred, hidden, context, score = las.speller.forward_step(rnn_in, hidden, encd)
        assert np.abs(raw_pred.cpu().numpy() - ref["logp"][s]).max() <= 1e-4
        assert np.abs(score[0].cpu().numpy() - ref["attn"][s]).max() <= 2e-5
        assert np.abs(context.cpu().numpy() - ref["context"][s]).max() <= 2e-5
        nxt = torch.nn.functional.one_hot(raw_pred.argmax(-1), c["V"]).float().unsqueeze(1)
        rnn_in = torch.cat([nxt, context.unsqueeze(1)], dim=-1)
    state = torch.randn(3, 1, 2 * c["H"], generator=g)
    score, ctx = las.speller.attention(state.cuda(), encd)
    psi = O.psi_project(enc.numpy().astype(np.float64), sd, np.float64)
    rs, rc = O.attention(state[:, 0].numpy().astype(np.float64), enc.numpy().astype(np.float64), psi, sd, np.float64)
    assert np.abs(score[0].cpu().numpy() - rs).max() <= 2e-6 and np.abs(ctx.cpu().numpy() - rc).max() <= 2e-6


def test_length_mask_extension_and_errors():
    c = tl.CONFIGS["tiny"]
    las = tl.build_model("tiny", max_label_len=4, seed=3, gain=3.0)
    sd = tl.state_dict_numpy(las)
    las = las.cuda()
    enc = torch.tanh(torch.randn(3, 8, 2 * c["H"], generator=torch.Generator().manual_seed(2)))
    lens = torch.tensor([8, 5, 1])
    ref = O.speller_forward(enc.numpy(), sd, c["sl"], 4, dtype=np.float64, enc_lengths=lens.numpy())
    preds, attns = las.speller(enc.cuda(), None, 0.0, enc_lengths=lens)
    attn = torch.stack([a[0] for a in attns]).cpu().numpy()
    assert np.abs(torch.stack(preds).cpu().numpy() - ref["logp"]).max() <= 1e-4
    assert np.array_equal(attn[:, 1, 5:], np.zeros_like(attn[:, 1, 5:]))  # masked steps get exactly zero weight
    # lengths == U reproduces the unmasked reference exactly
    p_full, _ = las.speller(enc.cuda(), None, 0.0, enc_lengths=torch.full((3,), 8))
    p_none, _ = las.speller(enc.cuda(), None, 0.0)
    assert torch.equal(torch.stack(p_full), torch.stack(p_none))
    # odd number of frames: the reference raises RuntimeError from view() (model/las_model.py:87)
    with pytest.raises(RuntimeError):
        las.listener(torch.randn(2, 30, 40, device="cuda"))  # 30 is not divisible by 4


def test_nll_sums_match_solver_loss():
    """'next' row f1: NLL(ignore_index=0) sums (solver/solver.py:62,70-77) computed on the device."""
    import ctypes as C

    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    S, B, V = 7, 5, 11
    g = torch.Generator().manual_seed(0)
    logp = torch.log_softmax(torch.randn(S, B, V, generator=g), -1).cuda()
    labels = torch.randint(0, V, (B, S), generator=g).to(torch.int32).cuda()
    out = torch.zeros(2, device="cuda")
    _cabi.check(lib.las_nll_sums(_cabi.ptr(logp), _cabi.ptr(labels), S, S, B, V, S, _cabi.ptr(out), _cabi.current_stream_ptr()))
    ref = O.nll_loss_ignore0(logp.permute(1, 0, 2).cpu().numpy().astype(np.float64), labels.cpu().numpy())
    assert abs(float(out[0] / out[1]) - ref) < 1e-5


def test_solver_batch_iterator_matches_oracle():
    """'next' row f1: solver.batch_iterator(is_training=False) -> (NLL(ignore_index=0) loss, per-utterance LER)."""
    from las_pytorch_b200.solver import batch_iterator

    c = tl.CONFIGS["small"]
    B, T, S = 5, 128, 20
    las = tl.build_model("small", max_label_len=S, seed=11, gain=3.0)
    sd = tl.state_dict_numpy(las)
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=11)
    labels[:, -3:] = 0  # padded tail, as collate_fn produces (utils/data.py:133-136)
    labels[:, -4] = 1   # <eos>
    ref = O.las_forward(x.numpy(), sd, c["L"], c["sl"], S, dtype=np.float64)
    ref_loss = O.nll_loss_ignore0(ref["logp"].transpose(1, 0, 2), labels.numpy())
    ref_ler = O.letter_error_rate(ref["tokens"].T, labels.numpy())
    loss, ler = batch_iterator(x.cuda(), tl.onehot(labels, c["V"]).cuda(), las.cuda(), None, 0.0, False, S, 0.1)
    assert abs(float(loss) - ref_loss) < 1e-4
    # the fused NLL terms equal the stand-alone reduction kernel over the returned log-probabilities
    from las_pytorch_b200.solver import nll_sums
    preds, _ = las(x.cuda(), None, 0.0, is_training=False, nll_labels=labels.cuda())
    sums = nll_sums(torch.stack(preds).contiguous(), labels.to(torch.int32).cuda(), S)
    terms = las.speller.last_nll_terms
    assert abs(float(terms.sum()) - float(sums[0])) < 1e-3 and int((terms != 0).sum()) == int(sums[1])
    if "bf16" in precisions():
        lasb = tl.build_model("small", max_label_len=S, seed=11, gain=3.0, precision="bf16").cuda()
        loss_b, _ = batch_iterator(x.cuda(), tl.onehot(labels, c["V"]).cuda(), lasb, None, 0.0, False, S, 0.1)
        assert abs(float(loss_b) - ref_loss) < 5e-2
    assert np.allclose(ler, ref_ler, atol=1e-12)
    with pytest.raises(NotImplementedError):
        batch_iterator(x.cuda(), tl.onehot(labels, c["V"]).cuda(), las, None, 0.9, True, S, 0.1)


@pytest.mark.parametrize("precision", precisions())
def test_reference_written_package_loads_and_decodes(precision):
    """Row f3 end to end: a package written by the REFERENCE (LAS.serialize + torch.save, model/las_model.py:42-63,
    train.py:181-192; generated by tests/golden/make_golden.py extras) is loaded with checkpoint.load_package -- plain and with
    nn.DataParallel's `module.` prefix -- moved to the GPU and decoded; outputs against what the reference computed from the very
    same module before saving it."""
    from las_pytorch_b200 import checkpoint

    g = np.load(os.path.join(tl.GOLDEN_DIR, "ref_package_tiny_outputs.npz"))
    tol = TOL[precision]
    for fname in ("ref_package_tiny.pth.tar", "ref_package_tiny_dataparallel.pth.tar"):
        las, pkg = checkpoint.load_package(os.path.join(tl.GOLDEN_DIR, fname), precision=precision, max_label_len=g["logp_greedy_f64"].shape[0])
        assert pkg["etype"] is torch.nn.LSTM and pkg["epoch"] == 7
        las = las.cuda()
        x, labels = torch.from_numpy(g["x"]), torch.from_numpy(g["labels"]).long()
        enc, logp, attn = run_ours(las, x, labels, las.speller.label_dim, "tf")
        assert np.abs(enc - g["enc_f64"]).max() <= tol["enc"]
        assert np.abs(logp - g["logp_tf_f64"]).max() <= tol["logp"]
        assert np.abs(attn - g["attn_tf_f64"]).max() <= tol["attn"]
        _, logp_g, _ = run_ours(las, x, labels, las.speller.label_dim, "greedy")
        if precision == "fp32":
            assert np.abs(logp_g - g["logp_greedy_f64"]).max() <= tol["logp"]
            assert np.array_equal(logp_g.argmax(-1), g["logp_greedy_f64"].argmax(-1))


def test_label_smoothing_and_nll_kernels_match_the_reference_values():
    """Row f1: las_label_smoothing_terms / las_nll_sums against numbers produced by the reference's own label_smoothing_loss and
    NLLLoss(ignore_index=0) (solver/solver.py:33-45,62; tests/golden/ref_solver_losses.npz)."""
    from las_pytorch_b200 import solver

    g = np.load(os.path.join(tl.GOLDEN_DIR, "ref_solver_losses.npz"))
    logp = torch.from_numpy(g["logp"]).cuda()          # [B,S,V]
    lab, lens = torch.from_numpy(g["labels"]).long(), g["lens"]
    V = logp.shape[-1]
    zero_pad = tl.onehot(lab, V).float()
    lab0 = lab.clone()
    for b, n in enumerate(lens):
        zero_pad[b, n:] = 0
        lab0[b, n:] = 0
    pad0 = tl.onehot(lab0, V).float()
    for ls in (0.1, 0.3):
        assert abs(float(solver.label_smoothing_loss(logp, zero_pad.cuda(), ls)) - float(g[f"ls_zero_pad_{ls}"])) < 2e-5
        assert abs(float(solver.label_smoothing_loss(logp, pad0.cuda(), ls)) - float(g[f"ls_pad0_{ls}"])) < 2e-5
    sums = solver.nll_sums(logp.permute(1, 0, 2).contiguous(), lab0.cuda().to(torch.int32).contiguous(), lab0.size(1))
    assert abs(float(sums[0] / sums[1]) - float(g["nll_ignore0"])) < 2e-5
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        solver.label_smoothing_loss(logp.cpu(), zero_pad, 0.1)


@pytest.mark.parametrize("precision", precisions())
def test_data_parallel_replicas_and_weight_updates(precision):
    """ADVICE r1 (high): the reference wraps the model in nn.DataParallel when device_count() > 1 (train.py:76-78).  Replicas share
    the original module's cache object and hold broadcast copies of the weights, so a cached kernel-layout image must never be
    reused across devices or across a weight update.  With two GPUs this runs the real nn.DataParallel; with one, replicate() +
    parallel_apply() place both replicas on cuda:0 (two host threads, same sharing of the cache)."""
    from torch.nn.parallel import parallel_apply, replicate

    c = tl.CONFIGS["small"]
    B, T, S = 6, 64, 8
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=83)
    las = tl.build_model("small", max_label_len=S, seed=83, gain=3.0, precision=precision).cuda(0)
    ndev = min(torch.cuda.device_count(), 2)

    def lone(model):
        return torch.stack(model(x.cuda(0), None, 0.0, False)[0]).cpu()

    def replicated(model):
        if ndev >= 2:
            out, _ = torch.nn.DataParallel(model, device_ids=[0, 1])(x.cuda(0), None, 0.0, False)
            return torch.stack(list(out)).cpu()
        reps = replicate(model, [0, 0])
        halves = parallel_apply(reps, [(x[:3].cuda(0), None, 0.0, False), (x[3:].cuda(0), None, 0.0, False)], devices=[0, 0])
        return torch.cat([torch.stack(list(h[0])) for h in halves], dim=1).cpu()

    for round_ in range(2):
        want = lone(las)
        for _ in range(2):
            got = replicated(las)
            if precision == "fp32":
                assert torch.equal(got, want)
            else:
                assert float((got - want).abs().max()) < 2e-2
        with torch.no_grad():  # an optimizer-style in-place update between calls: stale packed weights would reproduce `want`
            for p in las.parameters():
                p.mul_(1.5 if p.dim() == 2 else 1.0)
        assert float((lone(las) - want).abs().max()) > 1e-3
    # in-place writes through .data bypass the version counter: documented, with an explicit hook
    before = lone(las)
    for p in las.parameters():
        p.data.mul_(0.5)
    las.invalidate_packed_weights()
    assert float((lone(las) - before).abs().max()) > 1e-3


def test_mismatched_teacher_forcing_shapes_raise():
    """ADVICE r1 (medium): the kernels stride ground truth / labels by (B, label_dim); a mismatching tensor must raise like the
    reference's torch.cat (model/las_model.py:236) instead of reading out of bounds."""
    c = tl.CONFIGS["tiny"]
    las = tl.build_model("tiny", max_label_len=4, seed=3).cuda()
    enc = las.listener(torch.randn(3, 16, c["F"]).cuda())
    good = tl.onehot(torch.randint(2, c["V"], (3, 4)), c["V"]).cuda()
    np.random.seed(0)
    las.speller(enc, good, 1.1)
    for bad in (good[:2], torch.zeros(3, 4, c["V"] + 1, dtype=torch.int64).cuda()):
        np.random.seed(0)
        with pytest.raises(RuntimeError, match="ground_truth"):
            las.speller(enc, bad, 1.1)
    np.random.seed(0)
    with pytest.raises(RuntimeError, match="ground_truth"):
        las.speller(enc, torch.randint(2, c["V"], (2, 4)).cuda(), 1.1)
    with pytest.raises(RuntimeError, match="out of range"):
        np.random.seed(0)
        las.speller(enc, torch.full((3, 4), c["V"]), 1.1)
    with pytest.raises(RuntimeError, match="nll_labels"):
        las.speller(enc, None, 0.0, nll_labels=torch.zeros(2, 4, dtype=torch.int32).cuda())
    with pytest.raises(RuntimeError, match="enc_lengths"):
        las.speller(enc, None, 0.0, enc_lengths=torch.ones(2, dtype=torch.int32).cuda())


def test_solver_raises_when_the_decoder_is_shorter_than_the_labels():
    """ADVICE r1 (low): speller.max_label_len < label length made the fused loss silently too small; the reference fails with a
    shape error there (solver/solver.py:68-72)."""
    from las_pytorch_b200 import solver

    c = tl.CONFIGS["tiny"]
    las = tl.build_model("tiny", max_label_len=3, seed=3).cuda()
    x, labels = tl.make_inputs(2, 16, c["F"], 6, c["V"], seed=3)
    with pytest.raises(RuntimeError, match="max_label_len"):
        solver.batch_iterator(x.cuda(), tl.onehot(labels, c["V"]).cuda(), las, None, 0.0, False, 6, 0.0)


def _decode_kw(las, enc, steps, **kw):
    logp, attn, tok = las.speller._decode(enc, steps, **kw)
    torch.cuda.synchronize()
    return logp.clone(), attn.clone(), tok.clone()


@pytest.mark.parametrize("cfgname,B,T,S", [("small", 5, 64, 30), ("paper", 64, 320, 46), ("odd", 3, 48, 11)])
def test_bf16_segmented_decode_is_bit_identical(cfgname, B, T, S):
    """las_decode_io.segment_steps: the persistent decoder's step loop cut into several launches (what the serving pipeline and the
    <eos> early exit build on) carries h / c / context / fed-back word on the device and must reproduce the single launch bit for
    bit -- greedy, index and dense teacher forcing, raw feedback (decode_mode 0) and sampling."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS[cfgname]
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=91)
    for dm in (1, 0, 2):
        las = tl.build_model(cfgname, max_label_len=S, decode_mode=dm, seed=91, gain=3.0, precision="bf16").cuda()
        enc = las.listener(x.cuda())
        variants = [dict()]
        if dm == 1:
            variants += [dict(gt_index=labels.cuda().to(torch.int32).contiguous()),
                         dict(gt_dense=tl.onehot(labels, c["V"]).float().cuda().contiguous()),
                         dict(nll_labels=labels.cuda())]
        for kw in variants:
            torch.manual_seed(5)
            one = _decode_kw(las, enc, S, **kw)
            for seg in (2, 10, 16):
                torch.manual_seed(5)
                many = _decode_kw(las, enc, S, segment_steps=seg, **kw)
                for a, b in zip(one, many):
                    assert torch.equal(a, b), (cfgname, dm, list(kw), seg)


@pytest.mark.parametrize("cfgname,B,T,S", [("paper", 64, 320, 40), ("paper", 33, 160, 24), ("small", 47, 128, 30)])
def test_bf16_utterance_groups_equal_lockstep(cfgname, B, T, S):
    """Launches with more than 32 utterances run as two groups pipelined through the persistent decoder's LSTM CTAs (per-group
    counters, 32-row activation boxes, N = 32 MMAs: csrc/fast_speller.cu lstm_role_ts).  Every buffer is indexed by utterance row and a
    column's sum does not depend on N, so the outputs must equal the lockstep form (las_debug_set_option(19, 0)) bit for bit -- in
    every feedback mode, with length masks, segmented, and for group sizes 32 + 32, 32 + 1 and 32 + 15."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS[cfgname]
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=23)
    for dm in (1, 0, 2):
        las = tl.build_model(cfgname, max_label_len=S, decode_mode=dm, seed=23, gain=3.0, precision="bf16").cuda()
        enc = las.listener(x.cuda())
        U = enc.shape[1]
        lens = torch.tensor([U - (i % 7) for i in range(B)], dtype=torch.int32, device="cuda")
        variants = [dict(), dict(enc_lengths=lens), dict(segment_steps=10)]
        if dm == 1:
            variants += [dict(gt_index=labels.cuda().to(torch.int32).contiguous()),
                         dict(gt_dense=tl.onehot(labels, c["V"]).float().cuda().contiguous()),
                         dict(nll_labels=labels.cuda())]
        for kw in variants:
            outs = []
            for groups in (1, 0):
                lib.las_debug_set_option(19, groups)
                try:
                    torch.manual_seed(5)
                    outs.append(_decode_kw(las, enc, S, **kw))
                finally:
                    lib.las_debug_set_option(19, 1)
            for a, b in zip(*outs):
                assert torch.equal(a, b), (cfgname, B, dm, list(kw))


@pytest.mark.parametrize("precision", precisions())
def test_eos_early_exit(precision):
    """Row f4, <eos> early-exit batching (extension; the reference always runs max_label_len steps, model/las_model.py:205-209):
    decoding stops at the first check after every utterance has emitted <eos>; decoded steps equal the full decode, the rest is
    filled (<eos> tokens, zero log-probs / attention), steps_done says where it stopped.  No host synchronisation inside."""
    c = tl.CONFIGS["small"]
    B, T, S = 6, 64, 96
    las = tl.build_model("small", max_label_len=S, seed=97, gain=3.0, precision=precision).cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=97)
    enc = las.listener(x.cuda())
    logp, attn, tok = _decode_kw(las, enc, S)
    t = tok.cpu().numpy()
    # Free-running trajectories are utterance-specific, so build the batch from the utterances that DO emit a common token at
    # different times: <eos> := that token, the batch := those utterances repeated.
    best = None
    for v in range(c["V"]):
        first = np.where((t == v).any(0), (t == v).argmax(0), S)  # first step each utterance emits v
        utts = [b for b in range(B) if first[b] < S - 40]
        if len(utts) >= 2 and (best is None or len(utts) > len(best[1])):
            best = (v, utts)
    assert best is not None, f"no token is emitted by two utterances early enough; change the seed: {t.T.tolist()}"
    eos, utts = best
    x = x[[utts[i % len(utts)] for i in range(B)]]
    enc = las.listener(x.cuda())
    logp, attn, tok = _decode_kw(las, enc, S)
    t = tok.cpu().numpy()
    assert (t == eos).any(0).all()
    best = (eos, int((t == eos).argmax(0).max()) + 1)  # steps needed until every utterance has emitted <eos>
    eos, need = best
    for every in (8, 32):
        expect = min(S, -(-need // every) * every)
        las.speller.eos_token, las.speller.early_exit_every = eos, every
        preds, attns = las.speller(enc, None, 0.0, early_exit=True)
        torch.cuda.synchronize()
        assert int(las.speller.last_steps_done) == expect, (int(las.speller.last_steps_done), expect, need, every)
        lp, tk = torch.stack(preds), las.speller.last_tokens
        at = torch.stack([a[0] for a in attns])
        assert torch.equal(lp[:expect], logp[:expect]) and torch.equal(tk[:expect], tok[:expect]) and torch.equal(at[:expect], attn[:expect, 0])
        assert bool((tk[expect:] == eos).all()) and float(lp[expect:].abs().max() if expect < S else 0) == 0.0
        assert float(at[expect:].abs().max() if expect < S else 0) == 0.0
    # default stays the reference's behaviour: all max_label_len steps
    preds, _ = las.speller(enc, None, 0.0)
    assert torch.equal(torch.stack(preds), logp)
    # teacher forcing ignores the switch
    np.random.seed(0)
    labels = torch.randint(2, c["V"], (B, 12)).cuda()
    p1, _ = las.speller(enc, labels, 1.1, early_exit=True)
    assert len(p1) == 12


@pytest.mark.parametrize("cfgname,B,T,S,overlaps", [("paper", 64, 1600, 300, True), ("small", 32, 1600, 300, True), ("paper", 16, 3000, 600, True),
                                                    ("small", 4, 64, 12, True), ("odd", 3, 48, 6, None)])
def test_serving_pipeline_equals_forward(cfgname, B, T, S, overlaps):
    """LAS.serve(): batch i+1's listener under batch i's decoder (las_pipeline_step).  Every batch must get exactly what LAS.forward
    gives it on its own -- at the benchmarked shapes (c3, c2, c4), where the concurrent schedule applies, and at small / odd ones."""
    from las_pytorch_b200 import _cabi

    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    xs = [tl.make_inputs(B, T, c["F"], S, c["V"], seed=100 + i)[0].cuda() for i in range(4)]
    want = []
    for x in xs:
        preds, attns = las(x, None, 0.0, is_training=False)
        want.append((torch.stack(preds).clone(), torch.stack([a[0] for a in attns]).clone(), las.speller.last_tokens.clone()))
    if overlaps is not None:
        ld = _cabi.ListenerDims(B, T, c["F"], c["H"], c["L"], 0)
        sd = las.speller._dims(B, T >> c["L"], 2 * c["H"])
        import ctypes as C
        assert bool(_cabi.load_library().las_pipeline_overlaps(C.byref(ld), C.byref(sd), S, _cabi.MODE_BF16)) == overlaps
    for rounds in range(2):  # twice: the pipeline's workspaces / events are reused
        pipe = las.serve()
        got = []
        for x in xs:
            r = pipe.submit(x)
            if r is not None:
                got.append(r)
        got.append(pipe.flush())
        assert pipe.flush() is None
        torch.cuda.synchronize()
        assert len(got) == len(xs)
        for (lp, at, tk), r in zip(want, got):
            assert torch.equal(r.tokens, tk)
            assert torch.equal(r.logp, lp)
            assert torch.equal(r.attn, at)
            assert len(r.raw_pred_seq) == S and r.attention_record[0][0].shape == (B, T >> c["L"])


def test_serving_pipeline_fp32_and_masks_fall_back_to_the_same_results():
    c = tl.CONFIGS["small"]
    B, T, S = 4, 64, 10
    for precision in precisions():
        las = tl.build_model("small", max_label_len=S, seed=19, gain=3.0, precision=precision).cuda()
        xs = [tl.make_inputs(B, T, c["F"], S, c["V"], seed=200 + i)[0].cuda() for i in range(3)]
        lens = torch.tensor([64, 50, 33, 20])
        want = []
        for x in xs:
            preds, _ = las(x, None, 0.0, is_training=False, input_lengths=lens)
            want.append(torch.stack(preds).clone())
        pipe = las.serve(want_attention=False)
        got = [pipe.submit(x, input_lengths=lens) for x in xs][1:] + [pipe.flush()]
        torch.cuda.synchronize()
        for w, r in zip(want, got):
            assert torch.equal(r.logp, w) and r.attn is None


def test_bf16_results_do_not_depend_on_the_batch_an_utterance_is_in():
    """SURVEY.md 8e: the reference's output for an utterance is bitwise independent of how the batch is sharded, which is what
    multi-GPU sharding (bench.py --workload c5) relies on.  The listener picks its recurrence chunk (16 / 32 / 64 utterances per
    cluster) from the batch size: all variants must produce the same bits."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS["paper"]
    B, T = 40, 256
    lis = tl.build_model("paper", max_label_len=4, seed=17, gain=3.0, precision="bf16").listener.cuda()
    x, _ = tl.make_inputs(B, T, c["F"], 4, c["V"], seed=77)
    x = x.cuda()
    outs = []
    try:
        for bc in (16, 32, 64):
            lib.las_debug_set_option(9, bc)
            outs.append(lis(x).clone())
    finally:
        lib.las_debug_set_option(9, 0)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    parts = torch.cat([lis(x[:7]), lis(x[7:24]), lis(x[24:])], dim=0)
    assert torch.equal(parts, outs[0])


def test_bf16_generic_step_fused_equals_unfused_and_is_batch_independent():
    """The generic tensor-core decoder step (1024-wide cells, csrc/gen_step.cu) as one launch per stacked-cell layer + a cluster of CTAs
    per utterance for the attention, against the same step as separate GEMM / cell / operand kernels with one attention CTA per
    utterance (las_debug_set_option(12, 0)): the two sum in different orders, so they agree to fp32 round-off of the same bf16 products,
    not bit for bit.  The fused step picks its cluster size (8 / 4 / 2 / 1 CTAs per utterance) and its GEMM's N from the batch size:
    an utterance's result must not depend on either."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    c = tl.CONFIGS["shipped"]
    B, T, S = 80, 200, 8
    las = tl.build_model("shipped", max_label_len=S, seed=5, gain=2.0, precision="bf16").cuda()
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=5)
    enc = las.listener(x.cuda())
    lens = torch.tensor([enc.shape[1] - (i % 5) for i in range(B)], dtype=torch.int32, device="cuda")

    def run(e, **kw):
        torch.manual_seed(11)
        np.random.seed(0)
        preds, attns = las.speller(e, kw.pop("gt", None), kw.pop("rate", 0.0), **kw)
        return torch.stack(preds), torch.stack([a[0] for a in attns]), las.speller.last_tokens.clone()

    cases = {"greedy": dict(), "masked": dict(enc_lengths=lens), "index_tf": dict(gt=labels.cuda(), rate=1.1),
             "dense_tf": dict(gt=tl.onehot(labels, c["V"]).cuda(), rate=1.1)}
    fused = {k: run(enc, **dict(v)) for k, v in cases.items()}
    try:
        lib.las_debug_set_option(12, 0)
        unfused = {k: run(enc, **dict(v)) for k, v in cases.items()}
    finally:
        lib.las_debug_set_option(12, 1)
    # raw feedback (decode_mode 0), sampling (decode_mode 2) and the fused NLL terms go through the same operand-row outputs
    extra = {}
    for dm, kw in ((0, dict()), (2, dict()), (1, dict(nll_labels=labels[:16].cuda()))):
        m = tl.build_model("shipped", max_label_len=S, decode_mode=dm, seed=5, gain=2.0, precision="bf16").cuda()
        outs = []
        for opt in (1, 0):
            lib.las_debug_set_option(12, opt)
            try:
                torch.manual_seed(11)
                np.random.seed(0)
                preds, _ = m.speller(enc[:16].contiguous(), None, 0.0, **dict(kw))
                outs.append((torch.stack(preds), m.speller.last_tokens.clone(),
                             m.speller.last_nll_terms.clone() if kw else None))
            finally:
                lib.las_debug_set_option(12, 1)
        extra[dm if not kw else "nll"] = outs
    assert float((extra[0][0][0] - extra[0][1][0]).abs().max()) <= 5e-3          # raw: the log-probs themselves are fed back
    assert float((extra[2][0][1] == extra[2][1][1]).float().mean()) >= 0.9      # same counter-based draws unless a CDF edge moves
    assert float((extra["nll"][0][2] - extra["nll"][1][2]).abs().max()) <= 2e-3
    for k in cases:
        assert float((fused[k][0] - unfused[k][0]).abs().max()) <= 2e-3, k
        assert float((fused[k][1] - unfused[k][1]).abs().max()) <= 1e-3, k
        assert float((fused[k][2] == unfused[k][2]).float().mean()) >= 0.97, k
        assert float((fused[k][0].exp().sum(-1) - 1).abs().max()) < 1e-4 and float((fused[k][1].sum(-1) - 1).abs().max()) < 1e-4
    # masked encoder steps get exactly zero attention
    U = enc.shape[1]
    for b in (1, 4, 79):
        assert float(fused["masked"][1][:, b, U - (b % 5):].abs().max()) == 0.0
    # 3 utterances (8 CTAs each), 20 (4), 40 (2), 80 (1): the same bits
    for n in (3, 20, 40):
        part = run(enc[:n].contiguous())
        assert torch.equal(part[0], fused["greedy"][0][:, :n]) and torch.equal(part[1], fused["greedy"][1][:, :n]), n
    try:
        for cs in (1, 2, 4, 8):
            lib.las_debug_set_option(13, cs)
            part = run(enc[:16].contiguous())
            assert torch.equal(part[0], fused["greedy"][0][:, :16]), cs
    finally:
        lib.las_debug_set_option(13, 0)


@pytest.mark.parametrize("cfg,B", [
    (dict(F=40, H=20, L=2, sl=2, V=150, D=24, unit="GRU"), 5),          # Hs = 40: cells / K blocks / vocabulary none of them round
    (dict(F=40, H=36, L=2, sl=3, V=30, D=40, unit="RNN"), 19),          # one gate block, three layers, D not a multiple of 32
    (dict(F=40, H=44, L=2, sl=2, V=61, D=32, use_mlp=False), 33),       # no MLP in the attention (query = state), N = 48
    (dict(F=40, H=320, L=2, sl=1, V=30, D=64), 9),                      # LSTM too wide for the persistent decoder (Hs = 640), one layer
])
def test_bf16_generic_step_fused_equals_unfused_on_odd_shapes(cfg, B):
    """The fused generic step against the unfused one on shapes where nothing is a round number (hidden sizes that are not multiples of
    the 16-cell CTA slice or of the 64-column K block, vocabularies above the warp-level log-softmax, every cell type, the attention
    without its MLP): same bf16 products, different summation orders."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    from las_pytorch_b200 import _cabi

    lib = _cabi.load_library()
    T, S = 96, 7
    las = tl.build_model(cfg, max_label_len=S, seed=3, gain=2.0, precision="bf16").cuda()
    x, labels = tl.make_inputs(B, T, cfg["F"], S, cfg["V"], seed=3)
    enc = las.listener(x.cuda())
    U = enc.shape[1]
    lens = torch.tensor([max(1, U - (i % 4)) for i in range(B)], dtype=torch.int32, device="cuda")
    for kw in (dict(), dict(enc_lengths=lens), dict(gt=labels.cuda(), rate=1.1)):
        outs = []
        for opt in (1, 0):
            lib.las_debug_set_option(12, opt)
            try:
                np.random.seed(0)
                k = dict(kw)
                preds, attns = las.speller(enc, k.pop("gt", None), k.pop("rate", 0.0), **k)
                outs.append((torch.stack(preds), torch.stack([a[0] for a in attns])))
            finally:
                lib.las_debug_set_option(12, 1)
        # (an fp32 sum that differs in its last bit can round to the other bf16 neighbour; ungated tanh / GRU recurrences amplify that
        # 2^-9 step, the LSTM's gates damp it: DESIGN.md section 6)
        tol = 3e-3 if cfg.get("unit", "LSTM") == "LSTM" else 2e-2
        assert float((outs[0][0] - outs[1][0]).abs().max()) <= tol, (cfg, list(kw))
        assert float((outs[0][1] - outs[1][1]).abs().max()) <= tol / 2, (cfg, list(kw))
        assert float((outs[0][0].exp().sum(-1) - 1).abs().max()) < 1e-4


def test_large_batch_forward_is_chunk_pipelined_and_identical():
    """LAS.forward on a free-running batch larger than one decoder launch group (BASELINE config 5) runs chunk i+1's listener under
    chunk i's decoder; the outputs are bit for bit those of the plain path (forced by `--no-pipeline`-style separate calls)."""
    if "bf16" not in precisions():
        pytest.skip("bf16 mode not built")
    c = tl.CONFIGS["paper"]
    B, T, S = 150, 256, 16
    las = tl.build_model("paper", max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    x, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=123)
    x = x.cuda()
    assert las._chunk_pipelining_applies(x)
    np.random.seed(3)
    preds, attns = las(x, None, 0.0, is_training=False)
    drawn = np.random.random_sample()
    tok = las.speller.last_tokens.clone()
    # the plain path: whole-batch listener, then the decoder in its launch groups
    enc = las.listener(x)
    np.random.seed(3)
    p2, a2 = las.speller(enc, None, 0.0)
    assert np.random.random_sample() == drawn  # one draw from numpy's global RNG per call either way
    assert torch.equal(torch.stack(preds), torch.stack(p2))
    assert torch.equal(torch.stack([a[0] for a in attns]), torch.stack([a[0] for a in a2]))
    assert torch.equal(tok, las.speller.last_tokens) and tok.shape == (S, B)


@pytest.mark.parametrize("seed", list(range(24)))
def test_random_shapes_against_the_oracle(seed):
    """Randomised sweep over the shape space the persistent kernels select their variants from (hidden sizes / 64-wide atoms, batch
    sizes that leave TMEM lanes and warp slices empty, 1-3 speller layers, vocabularies up to the 64-wide word atom, encoder lengths
    across the single-CTA / split-attention boundary, odd step counts, segment lengths): both modes against the fp64 oracle,
    teacher-forced (index and one-hot) plus re-scored free-running decoding, segmented decode bit-identical to one launch."""
    rng = np.random.RandomState(1000 + seed)
    H = int(rng.choice([32, 64, 128, 256]))
    L = int(rng.choice([1, 2, 3]))
    sl = int(rng.choice([1, 2, 3]))
    V = int(rng.choice([5, 30, 42, 64]))
    D = int(rng.choice([16, 40, 64]))
    B = int(rng.choice([1, 3, 17, 33, 64]))
    U = int(rng.choice([3, 20, 70, 230, 300])) if H >= 128 else int(rng.choice([3, 20, 70]))
    if B * U * H > 64 * 120 * 256:  # keep the numpy oracle in seconds
        B = max(1, (64 * 120 * 256) // (U * H))
    T = U << L
    S = int(rng.choice([1, 2, 5, 9]))
    cfg = dict(F=40, H=H, L=L, sl=sl, V=V, D=D)
    x, labels = tl.make_inputs(B, T, cfg["F"], S, V, seed=seed)
    labels = labels % V
    ref = None
    for precision in precisions():
        las = tl.build_model(cfg, max_label_len=S, seed=seed, gain=2.5, precision=precision)
        sd = tl.state_dict_numpy(las)
        if ref is None:
            ref = O.las_forward(x.numpy(), sd, L, sl, S, ground_truth=labels.numpy(), teacher_forced=True, dtype=np.float64)
        las = las.cuda()
        tol = TOL[precision]
        for gt in (labels.cuda(), tl.onehot(labels, V).cuda()):
            np.random.seed(0)
            preds, attns = las(x.cuda(), gt, 1.1, is_training=True)
            logp = torch.stack(preds).cpu().numpy()
            attn = torch.stack([a[0] for a in attns]).cpu().numpy()
            assert np.abs(logp - ref["logp"]).max() <= tol["logp"], (cfg, B, U, S, precision)
            assert np.abs(attn - ref["attn"]).max() <= tol["attn"], (cfg, B, U, S, precision)
        preds, _ = las(x.cuda(), None, 0.0, is_training=False)
        logp_g = torch.stack(preds).cpu().numpy()
        tok = las.speller.last_tokens.cpu().numpy()
        assert np.array_equal(tok, logp_g.argmax(-1))
        rescored = O.las_forward(x.numpy(), sd, L, sl, S, ground_truth=tok.T, teacher_forced=True, dtype=np.float64)
        assert np.abs(logp_g - rescored["logp"]).max() <= tol["logp"], (cfg, B, U, S, precision)
        if precision != "fp32" and S >= 4:
            enc = las.listener(x.cuda())
            one = _decode_kw(las, enc, S)
            two = _decode_kw(las, enc, S, segment_steps=2)
            assert all(torch.equal(a, b) for a, b in zip(one, two)), (cfg, B, U, S)
