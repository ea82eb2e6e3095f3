"""Beam search's per-hypothesis attention (`return_attention`) against greedy decoding and the fp64 oracle, and its early exit
(`early_exit`) against the full run, bit for bit."""
import ctypes

import numpy as np
import pytest
import torch

from las_pytorch_b200 import _cabi
from oracle import las_oracle as O
from test_beam_search_gpu import LOGP_TOL, model_and_enc, rescore, tc_precisions, to_np, unfused_generic_step

pytestmark = pytest.mark.gpu

ATTN_TOL_FP32 = 2e-5  # the fp32 attention parity bound (DESIGN section 6)


def attention_bound(precision, sd, c, enc, r, enc_lengths, heads, ref):
    """fp32: the parity bound.  bf16 / fp16 (calibrated as DESIGN section 6 does): what rounding only the speller's 2-D weights to the
    operand format moves the oracle's attention on the same teacher-forced tokens, times 4, and at least the log-prob bound."""
    if precision == "fp32":
        return ATTN_TOL_FP32
    fmt = torch.bfloat16 if precision == "bf16" else torch.float16
    rounded = {k: (torch.from_numpy(np.asarray(v, np.float32)).to(fmt).float().numpy() if np.ndim(v) == 2 else v) for k, v in sd.items()}
    moved = np.abs(oracle_attention(enc, rounded, c, r, enc_lengths, heads) - ref)
    live = live_mask(r, heads)
    return max(LOGP_TOL[precision], 4 * float(np.where(live, moved, 0).max()))


def oracle_attention(enc, sd, c, r, enc_lengths, heads):
    """fp64 oracle attention of every returned hypothesis, teacher forced on its own tokens: the beam's shape [B,N,S,(heads,)U]."""
    B, N, S = r["tokens"].shape
    el = None if enc_lengths is None else np.repeat(enc_lengths, N)
    ref = O.speller_forward(np.repeat(enc, N, axis=0), sd, c["sl"], S, ground_truth=r["tokens"].reshape(B * N, S), dtype=np.float64,
                            enc_lengths=el)
    a = ref["attn"]  # [S, B*N, U] or [S, heads, B*N, U]
    U = a.shape[-1]
    if heads == 1:
        return a.transpose(1, 0, 2).reshape(B, N, S, U)
    return a.transpose(2, 0, 1, 3).reshape(B, N, S, heads, U)


def live_mask(r, heads):
    S = r["tokens"].shape[2]
    live = np.arange(S)[None, None, :] < r["lengths"][:, :, None]
    return live[..., None, None] if heads > 1 else live[..., None]


def greedy_attention(sp, e):
    """Speller.forward's attention record as [B, S, heads, U], its tokens [S, B]."""
    np.random.seed(0)
    _, rec = sp(e, ground_truth=None, teacher_force_rate=0.0)
    a = np.stack([np.stack([h.cpu().numpy() for h in step]) for step in rec])  # [S, heads, B, U]
    return a.transpose(2, 0, 1, 3), sp.last_tokens.cpu().numpy()


def check_width_one_alignment_is_greedy(cfg, precision):
    las, _, c, enc = model_and_enc(cfg, precision, B=3, U=20, S=16)
    sp = las.speller
    heads = sp.attention.multi_head
    e = torch.from_numpy(enc).cuda()
    g_attn, g_tok = greedy_attention(sp, e)
    r = to_np(sp.beam_search(e, beam_width=1, nbest=1, return_attention=True))
    a = r["attention"][:, 0]
    assert a.shape == ((3, 16, 20) if heads == 1 else (3, 16, heads, 20))
    if heads == 1:
        a = a[:, :, None, :]
    for b in range(enc.shape[0]):
        n = int(r["lengths"][b, 0])
        assert np.array_equal(r["tokens"][b, 0, :n], g_tok[:n, b])
        assert np.array_equal(a[b, :n], g_attn[b, :n]), (cfg, precision, b)
        assert np.all(a[b, n:] == 0)


@pytest.mark.parametrize("cfg", ["tiny", "odd", "tiny_mh", "tiny_nomlp", "tiny_gru", "tiny_rnn"])
def test_width_one_alignment_is_greedy_fp32(cfg):
    check_width_one_alignment_is_greedy(cfg, "fp32")


@pytest.mark.parametrize("precision", tc_precisions())
@pytest.mark.parametrize("cfg", ["tiny_gru", "tiny_rnn", "tiny_mh", "tiny_nomlp", "shipped"])
def test_width_one_alignment_is_greedy_tensor_core(cfg, precision):
    with unfused_generic_step():
        check_width_one_alignment_is_greedy(cfg, precision)


@pytest.mark.parametrize("precision", ["fp32"] + tc_precisions())
@pytest.mark.parametrize("cfg", ["tiny", "odd", "tiny_mh", "tiny_nomlp"])
def test_alignments_rescore_against_the_oracle(cfg, precision):
    las, sd, c, enc = model_and_enc(cfg, precision, B=4, U=16, S=18, scale=0.5)
    heads = las.speller.attention.multi_head
    lens = np.array([16, 7, 11, 3])
    for K, alpha, el in ((4, 0.0, None), (8, 0.8, lens)):
        r = to_np(las.speller.beam_search(torch.from_numpy(enc).cuda(), beam_width=K, nbest=K, length_penalty=alpha, return_attention=True,
                                          enc_lengths=None if el is None else torch.from_numpy(el).cuda()))
        B, N, S = r["tokens"].shape
        assert r["attention"].shape == ((B, N, S, 16) if heads == 1 else (B, N, S, heads, 16))
        live = np.arange(S)[None, None, :] < r["lengths"][:, :, None]
        assert np.abs(np.where(live, r["token_logp"] - rescore(enc, sd, c, r, el), 0)).max() <= LOGP_TOL[precision]  # same trajectory
        ref = oracle_attention(enc, sd, c, r, el, heads)
        lm = live_mask(r, heads)
        err = float(np.abs(np.where(lm, r["attention"] - ref, 0)).max())
        bound = attention_bound(precision, sd, c, enc, r, el, heads, ref)
        print(f"{cfg} {precision} K={K}: attention max-abs vs fp64 oracle {err:.2e} (bound {bound:.1e})")
        assert err <= bound, (cfg, precision, K, err, bound)
        assert np.all(np.where(lm, 0, r["attention"]) == 0)
        if el is not None:  # masked encoder steps get no weight
            masked = np.arange(16)[None, :] >= el[:, None]
            masked = masked[:, None, None, None, :] if heads > 1 else masked[:, None, None, :]
            assert np.all(np.where(np.broadcast_to(masked, r["attention"].shape), r["attention"], 0) == 0)


# ---- early exit -----------------------------------------------------------------------------------------------------------------

S_EE, EVERY = 24, 3  # a check period that is not even


def eos_biased(cfg, precision, bias):
    """A model whose <eos> logit is offset by `bias` (on tiny_mh +6 every hypothesis ends within 8 of the 24 steps; -30 makes <eos>
    unreachable)."""
    las, _, _, enc = model_and_enc(cfg, precision, B=4, U=12, S=S_EE)
    with torch.no_grad():
        las.speller.character_distribution.bias[1] += bias
    las.speller.early_exit_every = EVERY
    return las, enc


@pytest.mark.parametrize("precision", ["fp32"] + tc_precisions())
def test_early_exit_is_output_identical(precision):
    lens = torch.tensor([12, 5, 9, 3], dtype=torch.int32).cuda()
    stopped_early = []
    for cfg, bias in (("tiny_mh", 6.0), ("tiny", 3.0), ("tiny", -30.0)):
        las, enc = eos_biased(cfg, precision, bias)
        sp = las.speller
        sp.early_exit = True  # greedy decoding's switch: beam search ignores it
        e = torch.from_numpy(enc).cuda()
        for K in (1, 4, 8):
            for alpha in (0.0, 0.7):
                for el in (None, lens):
                    kw = dict(beam_width=K, nbest=K, length_penalty=alpha, enc_lengths=el, return_attention=True)
                    full = to_np(sp.beam_search(e, **kw))
                    sp.last_steps_done = None
                    early = to_np(sp.beam_search(e, early_exit=True, **kw))
                    for k in full:
                        assert np.array_equal(full[k], early[k]), (cfg, bias, K, alpha, el is not None, k)
                    done = int(sp.last_steps_done.item())
                    want = min(S_EE, -(-int(full["lengths"].max()) // EVERY) * EVERY)
                    assert done == want, (cfg, bias, K, alpha, done, want)
                    if bias < 0:
                        assert done == S_EE and np.all(full["lengths"] == S_EE)
                    stopped_early.append(done < S_EE)
    assert sum(stopped_early) >= len(stopped_early) // 3, stopped_early


def test_early_exit_does_not_change_a_default_call():
    las, enc = eos_biased("tiny", "fp32", 3.0)
    e = torch.from_numpy(enc).cuda()
    plain = to_np(las.speller.beam_search(e, beam_width=4, nbest=2))
    assert set(plain) == {"tokens", "lengths", "scores", "token_logp"}
    assert not hasattr(las.speller, "last_steps_done")
    early = to_np(las.speller.beam_search(e, beam_width=4, nbest=2, early_exit=True))
    assert all(np.array_equal(plain[k], early[k]) for k in plain)
    lp = to_np(las.beam_search(torch.zeros(4, 64, 40).cuda(), beam_width=4, nbest=2, return_attention=True, early_exit=True))
    assert lp["attention"].shape == (4, 2, S_EE, 64 >> 2)


def test_early_exit_under_graph_capture_is_refused_and_enqueues_nothing():
    las, enc = eos_biased("tiny", "fp32", 3.0)
    sp = las.speller
    e = torch.from_numpy(enc).cuda()
    sp.beam_search(e, beam_width=4, nbest=4, early_exit=True)  # packs the weights and allocates outside the capture
    torch.cuda.synchronize()
    lib = _cabi.load_library()
    # the C ABI on its own: LAS_EINVAL on a capturing stream, no launch
    buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    io = _cabi.BeamIO()
    io.enc, io.tokens, io.lengths, io.scores = (buf.data_ptr(),) * 4
    io.beam, io.nbest, io.eos_token, io.length_penalty = 4, 4, 1, 0.0
    io.early_exit, io.steps_done = 1, buf.data_ptr()
    dims = sp._dims(4, 12, 32)
    packed = sp._cache.packed[(0, ("beam", _cabi.MODE_FP32))][1]
    g = torch.cuda.CUDAGraph()
    lib.las_launch_count(1)
    with torch.cuda.graph(g):
        st = _cabi.current_stream_ptr()
        status = lib.las_speller_beam_search(ctypes.byref(io), ctypes.c_void_p(packed.data_ptr()), ctypes.byref(dims), S_EE, 0, 1,
                                             ctypes.c_void_p(buf.data_ptr()), buf.numel(), st)
        msg = lib.las_last_error()
        with pytest.raises(RuntimeError, match="captur"):
            sp.beam_search(e, beam_width=4, nbest=4, early_exit=True)
    assert status == -1 and b"captur" in msg, (status, msg)
    assert lib.las_launch_count(0) == 0
    # the same call outside the capture still runs
    r = to_np(sp.beam_search(e, beam_width=4, nbest=4, early_exit=True))
    assert r["lengths"].min() >= 1
