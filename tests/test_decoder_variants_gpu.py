"""Every decoder path against the fp64 oracle, at the shapes and settings that select it: attention without an activation
(mlp_activate_in_attention="None"), raw feedback (decode_mode 0) in every mode, and the generic tensor-core step at its real shapes.

Which path decodes a model is chosen by its shape and mode (csrc/las_api.cu speller_layout, speller_decode_f32):
  persistent  csrc/fast_speller.cu: tensor-core mode, LSTM, one head, MLP attention, Hs % 16 == 0 and <= 512, V <= 64
  fused       csrc/gen_step.cu cell step + attention (cluster kernel; attend_f32_kernel for multi-head): other tensor-core models, B <= 256
  unfused     build_a + GEMM + cell per layer, attend_f32_kernel: tensor-core models with B > 256, or las_debug_set_option(12, 0)
  fp32        lstm_cell_f32 per layer + the cluster kernel (attend_f32_kernel for multi-head or E % 4 != 0)
Each row of ROWS names its path, and the test asserts that path ran from the launches one more decoder step costs.

The speller is fed synthetic listener features, enc = tanh(randn(B, U, E)), so its shapes are free of the listener's limits.  Checks per
row: teacher forcing against the oracle; greedy decoding re-scored through the oracle on its own tokens; raw feedback re-scored with the
exact words the kernel fed back (its log-prob rows rounded to the 16-bit operand format); normalisation of log-probs and attention.
"""
import numpy as np
import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi
from oracle import las_oracle as O

pytestmark = pytest.mark.gpu

# the suite's parity bounds (tests/test_parity_gpu.py)
TOL = {"fp32": dict(enc=2e-5, logp=1e-4, attn=2e-5), "bf16": dict(enc=3e-2, logp=2e-2, attn=1e-2),
       "fp16": dict(enc=4e-3, logp=3e-3, attn=1.5e-3)}
OPERAND = {"bf16": torch.bfloat16, "fp16": torch.float16}

NONE = "None"
# name -> path, model (las_testlib config: H = Hs / 2), batch B, encoder steps U, feedback modes checked besides teacher forcing,
# whether to pass enc_lengths, weight gain, and las_debug_set_option(12, .) (0: the unfused generic step).  Cluster sizes of the
# attention kernel follow from B (gen_step.cu launch_attend_cluster; see test_fused_rows_cover_every_cluster_size).
ROWS = {
    # relu = 0 with W_phi in registers (D <= 64)
    "P1": dict(path="persistent", cfg=dict(H=32, sl=2, V=30, D=16, activate=NONE), B=5, U=20, feeds=("greedy",)),
    # relu = 0 with W_phi in shared memory (D > 64); 33 utterances = two utterance groups; masks.  (Gain 2: at 2.5 the energies of
    # this activation-free D = 128 attention are so peaked that the fp64 oracle itself, fed bf16-rounded weights and features, moves
    # by 1.9e-2 in the log-probs and 1.1e-2 in the attention, the whole bf16 bound; at gain 2 by 1.6e-3 and 8e-4.)
    "P2": dict(path="persistent", cfg=dict(H=64, sl=2, V=42, D=128, activate=NONE), B=33, U=70, feeds=("greedy",), lens=True, gain=2.0),
    # raw word through the dense word buffer; Hs = 80 is not a multiple of the 64-column atom
    "P3": dict(path="persistent", cfg=dict(H=40, sl=2, V=42, D=16), B=3, U=20, feeds=("raw",), gain=2.0),
    # split attention (2-CTA cluster per utterance: U = 300 at E = 512), no activation, raw word
    "P4": dict(path="persistent", cfg=dict(H=256, sl=2, V=30, D=64, activate=NONE), B=2, U=300, feeds=("raw",), gain=2.0),
    # the reference's shipped speller (1024-wide LSTM cells), with and without the activation
    "G1r": dict(path="fused", cfg=dict(H=512, sl=2, V=30, D=64), B=16, U=30, feeds=("greedy", "raw"), gain=2.0),
    "G1n": dict(path="fused", cfg=dict(H=512, sl=2, V=30, D=64, activate=NONE), B=16, U=30, feeds=("greedy", "raw"), gain=2.0),
    # GRU, V = 150: the block-wide log-softmax (V > 128); masks
    "G2": dict(path="fused", cfg=dict(H=20, sl=2, V=150, D=24, unit="GRU"), B=5, U=24, feeds=("greedy",), lens=True),
    # three RNN layers
    "G3": dict(path="fused", cfg=dict(H=36, sl=3, V=30, D=40, unit="RNN"), B=20, U=24, feeds=("greedy",)),
    # no MLP in the attention: query = state, keys = enc
    "G4": dict(path="fused", cfg=dict(H=44, sl=2, V=61, D=32, use_mlp=False), B=40, U=24, feeds=("greedy",)),
    # three heads, no activation: attend_f32_kernel writing the fused step's operand rows; masks
    "G5": dict(path="fused", cfg=dict(H=32, sl=2, V=30, D=24, heads=3, activate=NONE), B=80, U=20, feeds=("greedy",), lens=True),
    # an LSTM too wide for the persistent decoder, one layer
    "G6": dict(path="fused", cfg=dict(H=320, sl=1, V=30, D=64), B=9, U=24, feeds=("greedy",)),
    # more than 256 utterances: unfused, plain GEMM
    "U1": dict(path="unfused", cfg=dict(H=32, sl=2, V=30, D=16, unit="GRU"), B=300, U=12, feeds=("greedy", "raw")),
    # G2's model on the unfused step: swapped-operand GEMM (B <= 64) and plain GEMM
    "U2s": dict(path="unfused", cfg=dict(H=20, sl=2, V=150, D=24, unit="GRU"), B=5, U=24, feeds=("greedy",), lens=True, fused=0),
    "U2p": dict(path="unfused", cfg=dict(H=20, sl=2, V=150, D=24, unit="GRU"), B=80, U=24, feeds=("greedy",), lens=True, fused=0),
    # fp32: E = 38 (E % 4 != 0) selects attend_f32_kernel; E = 64 the cluster kernel
    "F1": dict(path="fp32", cfg=dict(H=19, sl=2, V=30, D=16, activate=NONE), B=5, U=20, feeds=("greedy", "raw")),
    "F2": dict(path="fp32", cfg=dict(H=32, sl=2, V=30, D=16, activate=NONE), B=5, U=20, feeds=("greedy",)),
}
S = 8


def tc_precisions():
    lib = _cabi.load_library()
    return [p for p, m in (("bf16", _cabi.MODE_BF16), ("fp16", _cabi.MODE_F16)) if lib.las_mode_available(m)]


def row_params(names):
    return [pytest.param(n, p, id=f"{n}-{p}") for n in names for p in (["fp32"] if ROWS[n]["path"] == "fp32" else tc_precisions())]


class debug_option:
    def __init__(self, key, value, default):
        self.key, self.value, self.default = key, value, default

    def __enter__(self):
        assert _cabi.load_library().las_debug_set_option(self.key, self.value) == 0

    def __exit__(self, *exc):
        assert _cabi.load_library().las_debug_set_option(self.key, self.default) == 0


def launches_per_step(row):
    """Kernel launches one more decoder step adds (speller_step): the fused generic step one per layer plus the attention, the unfused
    one a build_a + GEMM + cell per layer plus the attention, the fp32 step one cell kernel per layer plus the attention; the persistent
    decoder none (one launch runs every step)."""
    sl = row["cfg"]["sl"]
    return {"persistent": 0, "fused": sl + 1, "unfused": 3 * sl + 1, "fp32": sl + 1}[row["path"]]


def cluster_size(B, sms):
    """CTAs per utterance of the fused step's attention kernel (gen_step.cu launch_attend_cluster): at most half the SMs in all."""
    return next(c for c in (8, 4, 2, 1) if B * c <= sms // 2 or c == 1)


class Case:
    """One row in one precision: the model (on the GPU), its weights, the features, labels and lengths, and the oracle."""

    def __init__(self, name, precision, decode_mode=1):
        row = ROWS[name]
        self.row, self.precision = row, precision
        self.cfg = c = dict(F=40, L=1, **row["cfg"])
        self.B, self.U = row["B"], row["U"]
        self.act = c.get("activate", "relu") != NONE
        self.heads = c.get("heads", 1)
        seed = 1000 + sorted(ROWS).index(name)
        las = tl.build_model(c, max_label_len=S, decode_mode=decode_mode, seed=seed, gain=row.get("gain", 2.5), precision=precision)
        self.sd = tl.state_dict_numpy(las)
        self.sp = las.cuda().speller
        g = torch.Generator().manual_seed(seed)
        self.enc = torch.tanh(torch.randn(self.B, self.U, 2 * c["H"], generator=g))
        self.labels = torch.randint(2, c["V"], (self.B, S), generator=g)
        self.lens = None
        if row.get("lens"):
            self.lens = torch.tensor([max(1, self.U - (7 * b) % (self.U // 2)) for b in range(self.B)], dtype=torch.int32)
            assert int(self.lens.min()) < self.U
        self.encd = self.enc.cuda()
        self.lensd = None if self.lens is None else self.lens.cuda()

    def oracle(self, gt=None, decode_mode=1, rounded=False, repeat=1):
        """fp64 oracle, teacher forced on `gt` (indices [B,S] or dense [B,S,V]) or free running; `rounded`: the features and every 2-D
        weight rounded to the operand format first; `repeat`: each utterance `repeat` times in a row (beam hypotheses)."""
        enc, sd = np.repeat(self.enc.numpy(), repeat, axis=0), self.sd
        lens = None if self.lens is None else np.repeat(self.lens.numpy(), repeat)
        if rounded:
            fmt = OPERAND[self.precision]

            def rnd(a):
                return torch.from_numpy(np.asarray(a, np.float32)).to(fmt).float().numpy()

            enc, sd = rnd(enc), {k: (rnd(v) if v.ndim == 2 else v) for k, v in sd.items()}
        return O.speller_forward(enc, sd, self.cfg["sl"], S, ground_truth=gt, decode_mode=decode_mode, dtype=np.float64, enc_lengths=lens,
                                 activate=self.act)

    def bounds(self, gt, ref, repeat=1):
        """TOL of the mode; for GRU / RNN cells in the 16-bit modes at least 3x how far the oracle itself moves when its inputs and 2-D
        weights are rounded to the operand format (ungated recurrences amplify operand rounding far more than the LSTM)."""
        tol = dict(TOL[self.precision])
        if self.precision != "fp32" and self.cfg.get("unit", "LSTM") != "LSTM":
            rb = self.oracle(gt, rounded=True, repeat=repeat)
            for k in ("logp", "attn"):
                tol[k] = max(tol[k], 3.0 * float(np.abs(np.asarray(rb[k]) - np.asarray(ref[k])).max()))
        return tol

    def decode(self, gt=None):
        np.random.seed(0)
        preds, attns = self.sp(self.encd, None if gt is None else gt.cuda(), 1.1 if gt is not None else 0.0, enc_lengths=self.lensd)
        logp = torch.stack(preds).cpu().numpy()
        attn = torch.stack([torch.stack(list(a)) for a in attns]).cpu().numpy()  # [S, heads, B, U]
        return logp, attn, self.sp.last_tokens.cpu().numpy()

    def check(self, logp, attn, ref, tol, what):
        ra = np.asarray(ref["attn"])
        ra = ra[:, None] if self.heads == 1 else ra  # [S, heads, B, U]
        err_l, err_a = float(np.abs(logp - ref["logp"]).max()), float(np.abs(attn - ra).max())
        print(f"{what}: log-prob err {err_l:.2e} (bound {tol['logp']:.1e}), attention err {err_a:.2e} (bound {tol['attn']:.1e})")
        assert err_l <= tol["logp"], (what, err_l, tol["logp"])
        assert err_a <= tol["attn"], (what, err_a, tol["attn"])
        assert np.abs(np.exp(logp).sum(-1) - 1).max() < 1e-4, what
        assert np.abs(attn.sum(-1) - 1).max() < 1e-4, what
        if self.lens is not None:
            for b, n in enumerate(self.lens.tolist()):
                assert np.all(attn[:, :, b, n:] == 0), (what, b)  # masked frames get exactly zero weight

    def assert_path(self):
        lib = _cabi.load_library()
        counts = []
        for steps in (4, 12):
            self.sp._decode(self.encd, steps, enc_lengths=self.lensd)  # packs the weights on the first call
            torch.cuda.synchronize()
            lib.las_launch_count(1)
            self.sp._decode(self.encd, steps, enc_lengths=self.lensd)
            torch.cuda.synchronize()
            counts.append(int(lib.las_launch_count(0)))
        assert counts[1] - counts[0] == 8 * launches_per_step(self.row), (self.row["path"], counts)
        if self.row["path"] == "persistent":
            assert counts[1] < 12, counts  # fewer launches than steps


@pytest.mark.parametrize("name,precision", row_params(ROWS))
def test_decoder_path_against_the_oracle(name, precision):
    row = ROWS[name]
    with debug_option(12, row.get("fused", 1), 1):
        case = Case(name, precision)
        case.assert_path()
        # teacher forcing with index labels
        ref = case.oracle(case.labels.numpy())
        logp, attn, _ = case.decode(case.labels)
        case.check(logp, attn, ref, case.bounds(case.labels.numpy(), ref), f"{name} {precision} teacher forced")
        if "greedy" in row["feeds"]:
            logp, attn, tok = case.decode()
            assert np.array_equal(tok, logp.argmax(-1))
            ref = case.oracle(tok.T)  # every step's log-probs are the oracle's for the tokens that were fed back
            case.check(logp, attn, ref, case.bounds(tok.T, ref), f"{name} {precision} greedy, re-scored")
        if "raw" in row["feeds"]:
            raw = Case(name, precision, decode_mode=0)
            raw.assert_path()
            logp, attn, tok = raw.decode()
            assert np.array_equal(tok, logp.argmax(-1))
            # The word fed back after step s is log-prob row s, rounded to the operand format in the tensor-core modes: as dense ground
            # truth it makes the oracle see exactly the kernel's inputs.
            fed = logp if precision == "fp32" else torch.from_numpy(logp).to(OPERAND[precision]).float().numpy()
            gt = fed.transpose(1, 0, 2).astype(np.float64)
            ref = raw.oracle(gt)
            raw.check(logp, attn, ref, raw.bounds(gt, ref), f"{name} {precision} raw, re-scored")
            if precision == "fp32":
                free = raw.oracle(decode_mode=0)
                raw.check(logp, attn, free, TOL["fp32"], f"{name} fp32 raw, free running")


def test_fused_rows_cover_every_cluster_size():
    """The fused rows' batch sizes select every cluster size of the attention kernel (8 / 4 / 2 / 1 CTAs per utterance) on this device."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sizes = {cluster_size(r["B"], sms) for r in ROWS.values() if r["path"] == "fused" and r["cfg"].get("heads", 1) == 1}
    assert sizes == {8, 4, 2, 1}, (sms, sizes)


# ---- beam search (the launch-per-step form: the unfused generic step in the tensor-core modes) ---------------------------------------

def beam_rescore(case, r):
    """Oracle log-probs and attention of every returned hypothesis, teacher forced on its own tokens: [B,N,S], [B,N,S,U]."""
    B, N, _ = r["tokens"].shape
    gt = r["tokens"].reshape(B * N, S)
    ref = case.oracle(gt, repeat=N)
    lp = ref["logp"][np.arange(S)[:, None], np.arange(B * N)[None, :], gt.T].T.reshape(B, N, S)
    return lp, ref["attn"].transpose(1, 0, 2).reshape(B, N, S, -1), case.bounds(gt, ref, repeat=N), ref


def to_np(r):
    torch.cuda.synchronize()
    return {k: getattr(r, k).cpu().numpy() for k in r._fields}


@pytest.mark.parametrize("name,precision", row_params(["P1", "G2", "G4"]))
def test_beam_width_one_is_greedy(name, precision):
    case = Case(name, precision)
    sp = case.sp
    if ROWS[name]["path"] == "persistent":
        # greedy decoding of this model runs on the persistent decoder, beam search on the generic step: different operand sums, so the
        # check is that each chosen token is the oracle's argmax wherever the oracle's top-2 margin exceeds twice the log-prob bound
        r = to_np(sp.beam_search(case.encd, beam_width=1, nbest=1, enc_lengths=case.lensd))
        lp, _, tol, ref = beam_rescore(case, r)
        n = r["lengths"][:, 0]
        live = np.arange(S)[None, :] < n[:, None]
        assert np.abs(np.where(live, r["token_logp"][:, 0] - lp[:, 0], 0)).max() <= tol["logp"]
        srt = np.sort(ref["logp"], axis=-1)
        safe = ((srt[..., -1] - srt[..., -2]) > 2 * tol["logp"]).T & live
        assert np.array_equal(r["tokens"][:, 0][safe], ref["logp"].argmax(-1).T[safe])
        assert safe.sum() >= 0.5 * live.sum(), (safe.sum(), live.sum())
        return
    with debug_option(12, 0, 1):  # greedy decoding on the unfused step and one-CTA attention kernel, which beam search runs on too
        np.random.seed(0)
        _, rec = sp(case.encd, None, 0.0, enc_lengths=case.lensd)
        g_tok, g_lp = sp.last_tokens.cpu().numpy(), sp.last_logp.cpu().numpy()
        g_attn = np.stack([a[0].cpu().numpy() for a in rec])  # [S, B, U]
        r = to_np(sp.beam_search(case.encd, beam_width=1, nbest=1, enc_lengths=case.lensd, return_attention=True))
    for b in range(case.B):
        hit = np.nonzero(g_tok[:, b] == 1)[0]
        n = hit[0] + 1 if len(hit) else S
        assert r["lengths"][b, 0] == n
        assert np.array_equal(r["tokens"][b, 0, :n], g_tok[:n, b])
        assert np.array_equal(r["token_logp"][b, 0, :n], g_lp[np.arange(n), b, g_tok[:n, b]])
        assert np.array_equal(r["attention"][b, 0, :n], g_attn[:n, b])


@pytest.mark.parametrize("name,precision", row_params(["P1", "G2", "G4"]))
def test_beam_hypotheses_rescore_against_the_oracle(name, precision):
    case = Case(name, precision)
    r = to_np(case.sp.beam_search(case.encd, beam_width=4, nbest=2, return_attention=True, enc_lengths=case.lensd))
    lp, attn, tol, _ = beam_rescore(case, r)
    live = np.arange(S)[None, None, :] < r["lengths"][:, :, None]
    err_l = float(np.abs(np.where(live, r["token_logp"] - lp, 0)).max())
    err_a = float(np.abs(np.where(live[..., None], r["attention"] - attn, 0)).max())
    print(f"{name} {precision} beam: token log-prob err {err_l:.2e} (bound {tol['logp']:.1e}), attention err {err_a:.2e} "
          f"(bound {tol['attn']:.1e})")
    assert err_l <= tol["logp"] and err_a <= tol["attn"], (err_l, err_a, tol)
    assert np.all(np.where(live[..., None], 0, r["attention"]) == 0)
    if case.lens is not None:
        for b, n in enumerate(case.lens.tolist()):
            assert np.all(r["attention"][b, :, :, n:] == 0)


# ---- Attention.forward ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("heads", [1, 3])
@pytest.mark.parametrize("H", [16, 19])  # E = 32 and E = 38 (E % 4 != 0)
def test_attention_api_without_activation(H, heads):
    cfg = dict(F=40, H=H, L=1, sl=1, V=30, D=8, heads=heads, activate=NONE)
    las = tl.build_model(cfg, max_label_len=3, seed=9, gain=2.5)
    sd = {k: v.astype(np.float64) for k, v in tl.state_dict_numpy(las).items()}
    las = las.cuda()
    g = torch.Generator().manual_seed(2)
    enc = torch.tanh(torch.randn(3, 8, 2 * H, generator=g))
    state = torch.randn(3, 1, 2 * H, generator=g)
    score, ctx = las.speller.attention(state.cuda(), enc.cuda())
    e64 = enc.numpy().astype(np.float64)
    psi = O.psi_project(e64, sd, np.float64, activate=False)
    rs, rc = O.attention(state[:, 0].numpy().astype(np.float64), e64, psi, sd, np.float64, activate=False)
    rs = rs if heads > 1 else [rs]
    assert len(score) == heads
    for s_h, r_h in zip(score, rs):
        assert np.abs(s_h.cpu().numpy() - r_h).max() <= 2e-6
    assert np.abs(ctx.cpu().numpy() - rc).max() <= 2e-6
