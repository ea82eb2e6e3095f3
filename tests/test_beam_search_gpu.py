"""Beam search on the device (las_speller_beam_search) against greedy decoding, the fp64 reference in test_beam_search_cpu.py, itself
across batch sizes, and its output contract."""
import numpy as np
import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi
from oracle import las_oracle as O
from test_beam_search_cpu import speller_beam_search

pytestmark = pytest.mark.gpu

LOGP_TOL = {"fp32": 1e-4, "bf16": 2e-2, "fp16": 3e-3}


def tc_precisions():
    lib = _cabi.load_library()
    return [p for p, m in (("bf16", _cabi.MODE_BF16), ("fp16", _cabi.MODE_F16)) if lib.las_mode_available(m)]


class unfused_generic_step:
    """las_debug_set_option(12, 0): the greedy tensor-core decoder takes the step-per-launch path that beam search runs on."""

    def __enter__(self):
        assert _cabi.load_library().las_debug_set_option(12, 0) == 0

    def __exit__(self, *exc):
        assert _cabi.load_library().las_debug_set_option(12, 1) == 0


def model_and_enc(cfg, precision, B, U, S, seed=31, gain=3.0, scale=2.0):
    las = tl.build_model(cfg, max_label_len=S, seed=seed, gain=gain, precision=precision)
    c = tl.CONFIGS[cfg]
    enc = np.random.RandomState(seed).standard_normal((B, U, 2 * c["H"])).astype(np.float32) * scale
    return las.cuda(), tl.state_dict_numpy(las), c, enc


def to_np(r):
    torch.cuda.synchronize()
    return {k: getattr(r, k).cpu().numpy() for k in r._fields}


def check_width_one_is_greedy(cfg, precision):
    las, _, c, enc = model_and_enc(cfg, precision, B=3, U=20, S=16)
    sp = las.speller
    e = torch.from_numpy(enc).cuda()
    np.random.seed(0)
    sp(e, ground_truth=None, teacher_force_rate=0.0)
    g_tok, g_lp = sp.last_tokens.cpu().numpy(), sp.last_logp.cpu().numpy()
    r = to_np(sp.beam_search(e, beam_width=1, nbest=1))
    for b in range(enc.shape[0]):
        hit = np.nonzero(g_tok[:, b] == 1)[0]
        n = hit[0] + 1 if len(hit) else g_tok.shape[0]
        assert r["lengths"][b, 0] == n
        assert np.array_equal(r["tokens"][b, 0, :n], g_tok[:n, b])
        assert np.array_equal(r["token_logp"][b, 0, :n], g_lp[np.arange(n), b, g_tok[:n, b]])


@pytest.mark.parametrize("cfg", ["tiny", "odd", "tiny_mh", "tiny_nomlp", "tiny_gru", "tiny_rnn"])
def test_width_one_is_greedy_fp32(cfg):
    check_width_one_is_greedy(cfg, "fp32")


@pytest.mark.parametrize("precision", tc_precisions())
@pytest.mark.parametrize("cfg", ["tiny_gru", "tiny_rnn", "tiny_mh", "tiny_nomlp", "shipped"])
def test_width_one_is_greedy_tensor_core(cfg, precision):
    with unfused_generic_step():
        check_width_one_is_greedy(cfg, precision)


@pytest.mark.parametrize("cfg", ["tiny", "odd", "tiny_gru", "tiny_mh"])
def test_fp32_matches_the_fp64_reference(cfg):
    B, U = 6, 12
    # (a GRU at gain 3 fed scale-2 features is chaotic: fp32 round-off alone moves its scores by 1e-4 per step)
    las, sd, c, enc = model_and_enc(cfg, "fp32", B=B, U=U, S=20, scale=0.5 if cfg == "tiny_gru" else 2.0)
    lens = np.array([12, 5, 9, 1, 12, 7])
    compared = safe_total = 0
    for K in (2, 4, 8):
        S = 12 + K
        for el in (None, lens):
            ref = speller_beam_search(enc, sd, c["sl"], S, K, K, enc_lengths=el)
            r = to_np(las.speller.beam_search(torch.from_numpy(enc).cuda(), beam_width=K, nbest=K, max_steps=S,
                                              enc_lengths=None if el is None else torch.from_numpy(el).cuda()))
            safe = ref["margins"] > 1e-3
            compared += B
            safe_total += int(safe.sum())
            assert np.array_equal(r["tokens"][safe], ref["tokens"][safe]), (K, el)
            assert np.array_equal(r["lengths"][safe], ref["lengths"][safe]), (K, el)
            assert np.abs(r["scores"][safe] - ref["scores"][safe]).max(initial=0) <= 1e-4 * S
    assert safe_total >= 0.6 * compared, (safe_total, compared)


def rescore(enc, sd, c, r, enc_lengths=None):
    """Oracle log-probs (fp64) of every returned hypothesis's own tokens, teacher forced: [B, N, S]."""
    B, N, S = r["tokens"].shape
    gt = r["tokens"].reshape(B * N, S)
    el = None if enc_lengths is None else np.repeat(enc_lengths, N)
    ref = O.speller_forward(np.repeat(enc, N, axis=0), sd, c["sl"], S, ground_truth=gt, dtype=np.float64, enc_lengths=el)
    lp = ref["logp"][np.arange(S)[:, None], np.arange(B * N)[None, :], gt.T]  # [S, B*N]
    return lp.T.reshape(B, N, S)


def check_output_contract(r, alpha, eos=1):
    B, N, S = r["tokens"].shape
    for b in range(B):
        keys = []
        hyps = set()
        for n in range(N):
            L = int(r["lengths"][b, n])
            assert np.all(r["tokens"][b, n, L:] == eos) and np.all(r["token_logp"][b, n, L:] == 0)
            if L == 0:
                assert r["scores"][b, n] == -np.inf
                keys.append(-np.inf)
                continue
            hit = np.nonzero(r["tokens"][b, n] == eos)[0]
            assert L == (hit[0] + 1 if len(hit) else S)
            assert r["scores"][b, n] == np.add.accumulate(r["token_logp"][b, n].astype(np.float32))[-1]
            keys.append(np.float32(r["scores"][b, n]) / np.power(np.float32(L), np.float32(alpha)))
            hyps.add(tuple(r["tokens"][b, n, :L]))
        assert len(hyps) == sum(1 for k in keys if k != -np.inf), "duplicate hypotheses"
        keys = np.array(keys)
        assert np.all(keys[:-1] >= keys[1:] - 1e-6 * np.abs(keys[1:])), keys


@pytest.mark.parametrize("precision", ["fp32"] + tc_precisions())
def test_rescoring_and_output_contract_on_tiny_models(precision):
    tol = LOGP_TOL[precision]
    for cfg in ("tiny", "odd"):
        las, sd, c, enc = model_and_enc(cfg, precision, B=4, U=16, S=18, scale=0.5)
        lens = np.array([16, 7, 11, 3])
        for K, alpha, el in ((4, 0.0, None), (8, 0.8, lens)):
            r = to_np(las.speller.beam_search(torch.from_numpy(enc).cuda(), beam_width=K, nbest=K, length_penalty=alpha,
                                              enc_lengths=None if el is None else torch.from_numpy(el).cuda()))
            check_output_contract(r, alpha)
            lp = rescore(enc, sd, c, r, el)
            live = np.arange(r["tokens"].shape[2])[None, None, :] < r["lengths"][:, :, None]
            assert np.abs(np.where(live, r["token_logp"] - lp, 0)).max() <= tol, (cfg, K)


@pytest.mark.parametrize("precision", ["fp32"] + tc_precisions())
def test_paper_model_rescored(precision):
    """The paper model (persistent-decoder shape in the tensor-core modes) runs through the beam pack's generic layout."""
    c = tl.CONFIGS["paper"]
    B, T, S, K = 8, 800, 60, 4
    las = tl.build_model("paper", max_label_len=S, seed=7, precision=precision).cuda()
    sd = tl.state_dict_numpy(las)
    x, _ = tl.make_inputs(B, T, c["F"], 4, c["V"], seed=7)
    x = x.cuda()
    r = to_np(las.beam_search(x, beam_width=K, nbest=K))
    enc = las.listener(x).cpu().numpy()
    check_output_contract(r, 0.0)
    lp = rescore(enc, sd, c, r)
    live = np.arange(S)[None, None, :] < r["lengths"][:, :, None]
    assert np.abs(np.where(live, r["token_logp"] - lp, 0)).max() <= LOGP_TOL[precision]


def test_nbest_is_a_prefix_of_the_full_beam():
    las, _, _, enc = model_and_enc("tiny", "fp32", B=5, U=12, S=16)
    e = torch.from_numpy(enc).cuda()
    for alpha in (0.0, 1.0):
        full = to_np(las.speller.beam_search(e, beam_width=8, nbest=8, length_penalty=alpha))
        for n in (1, 3):
            part = to_np(las.speller.beam_search(e, beam_width=8, nbest=n, length_penalty=alpha))
            for k in full:
                assert np.array_equal(part[k], full[k][:, :n]), (alpha, n, k)


def beam_rows(las, enc, K=4, S=16):
    return to_np(las.speller.beam_search(torch.from_numpy(enc).cuda(), beam_width=K, nbest=K, max_steps=S))


def same(a, b, idx):
    return all(np.array_equal(a[k], b[k][idx]) for k in a)


def test_batch_independence_fp32():
    las, _, _, enc = model_and_enc("tiny", "fp32", B=64, U=12, S=16)
    r64 = beam_rows(las, enc)
    r1 = beam_rows(las, enc[:1])
    r3 = beam_rows(las, enc[:3])
    assert same(r1, r64, slice(0, 1)) and same(r3, r64, slice(0, 3))


@pytest.mark.parametrize("precision", tc_precisions())
def test_batch_independence_tensor_core(precision):
    """The generic step's GEMM changes orientation at 64 decoder rows: bit-identity on each side, round-off agreement across."""
    las, _, _, enc = model_and_enc("tiny", precision, B=64, U=12, S=16)
    small = {n: beam_rows(las, enc[:n]) for n in (1, 3, 16)}      # 4, 12 and 64 rows
    large = {n: beam_rows(las, enc[:n]) for n in (17, 64)}        # 68 and 256 rows
    assert same(small[1], small[16], slice(0, 1)) and same(small[3], small[16], slice(0, 3))
    assert same(large[17], large[64], slice(0, 17))
    a, b = small[16], {k: v[:16] for k, v in large[64].items()}
    agree = np.all(a["tokens"] == b["tokens"], axis=(1, 2))
    assert agree.mean() >= 0.5, agree
    assert np.abs(a["token_logp"][agree] - b["token_logp"][agree]).max(initial=0) <= 2e-3
    print(f"{precision}: 16 utterances across the GEMM switch bit-identical: {same(a, b, slice(None))}")


def test_no_side_effects_on_rngs_caches_or_greedy_decoding():
    precision = (tc_precisions() or ["fp32"])[0]
    las, _, c, _ = model_and_enc("tiny", precision, B=1, U=1, S=12)
    x, _ = tl.make_inputs(3, 64, c["F"], 4, c["V"], seed=3)
    x = x.cuda()
    np.random.seed(0)
    before = [t.cpu().numpy() for t in torch.stack(las(x, None, 0.0, is_training=False)[0])]
    np_state, torch_state, cuda_state = np.random.get_state(), torch.get_rng_state(), torch.cuda.get_rng_state()
    las.beam_search(x, beam_width=4, nbest=2)
    torch.cuda.synchronize()
    assert np.array_equal(np.random.get_state()[1], np_state[1]) and np.random.get_state()[2] == np_state[2]
    assert torch.equal(torch.get_rng_state(), torch_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    np.random.seed(0)
    after = [t.cpu().numpy() for t in torch.stack(las(x, None, 0.0, is_training=False)[0])]
    assert all(np.array_equal(p, q) for p, q in zip(before, after))
    mode = _cabi.MODE_FP32 if precision == "fp32" else (_cabi.MODE_BF16 if precision == "bf16" else _cabi.MODE_F16)
    dev = x.device.index
    assert {(dev, mode), (dev, ("beam", mode))} <= set(las.speller._cache.packed)  # greedy and beam packs side by side
