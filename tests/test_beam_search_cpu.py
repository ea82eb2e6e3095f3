"""Beam search without a GPU: the numpy reference against greedy decoding and a brute-force n-best, and the argument checks of the C
ABI and of the Python API.  `speller_beam_search` is the reference the GPU tests (test_beam_search_gpu.py) compare against."""
import ctypes
import math

import numpy as np
import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi
from oracle import las_oracle as O


def speller_beam_search(enc, sd, num_layers, steps, beam, nbest, eos=1, length_penalty=0.0, dtype=np.float64, enc_lengths=None,
                        prefix="speller"):
    """Beam search as include/las_b200.h defines it, on top of the oracle's decoder step.  K = beam rows per utterance, all starting
    in the reference's initial state; only row 0 is live.  Per step a live row k offers (k, v, score[k] + logp[k, v]), a finished row
    (k, eos, score[k]) with log-prob 0; the K best by (score desc, parent asc, token asc) become the new rows.  The K final rows are
    ranked by score / length**length_penalty (ties: lower slot).  Returns dict(tokens [B,N,S], token_logp [B,N,S], lengths [B,N],
    scores [B,N], margins [B], min_margin): margins[b] is the smallest gap, over the steps and the final ranking of utterance b, between
    the K-th kept and the best dropped candidate, and between consecutive ranks among the first N + 1 final keys."""
    enc = np.asarray(enc, dtype=dtype)
    B, U, E = enc.shape
    K, S = beam, steps
    w_cd = O._w(sd, f"{prefix}.character_distribution.weight", dtype)
    b_cd = O._w(sd, f"{prefix}.character_distribution.bias", dtype)
    V = w_cd.shape[0]
    hs = O._w(sd, f"{prefix}.rnn_layer.weight_hh_l0", dtype).shape[1]
    psi = O.psi_project(enc, sd, dtype, prefix) if f"{prefix}.attention.psi.weight" in sd else enc
    enc_r, psi_r = np.repeat(enc, K, axis=0), np.repeat(psi, K, axis=0)  # row b*K + k attends over utterance b
    len_r = None if enc_lengths is None else np.repeat(np.asarray(enc_lengths), K)
    h = [np.zeros((B * K, hs), dtype=dtype) for _ in range(num_layers)]
    c = [np.zeros((B * K, hs), dtype=dtype) for _ in range(num_layers)]
    word = np.zeros((B * K, V), dtype=dtype)
    word[:, 0] = 1
    ctx = enc_r[:, 0, :].copy()
    score = np.full((B, K), -np.inf, dtype=dtype)
    score[:, 0] = 0
    fin = np.zeros((B, K), dtype=bool)
    hist_tok = np.full((B, K, S), eos, dtype=np.int64)
    hist_lp = np.zeros((B, K, S), dtype=dtype)
    margins = np.full(B, np.inf)
    for s in range(S):
        inp = np.concatenate([word, ctx], axis=-1)
        for l in range(num_layers):
            px = inp @ O._w(sd, f"{prefix}.rnn_layer.weight_ih_l{l}", dtype).T + O._w(sd, f"{prefix}.rnn_layer.bias_ih_l{l}", dtype)
            ph = h[l] @ O._w(sd, f"{prefix}.rnn_layer.weight_hh_l{l}", dtype).T + O._w(sd, f"{prefix}.rnn_layer.bias_hh_l{l}", dtype)
            h[l], c[l] = O.rnn_cell_step(px, ph, h[l], c[l])
            inp = h[l]
        _, ctx = O.attention(h[-1], enc_r, psi_r, sd, dtype, prefix, enc_lengths=len_r)
        logp = O.log_softmax(np.concatenate([h[-1], ctx], axis=-1) @ w_cd.T + b_cd).astype(dtype).reshape(B, K, V)
        perm = np.zeros(B * K, dtype=np.int64)
        new_tok = np.full((B, K), eos, dtype=np.int64)
        for b in range(B):
            vals, par, tok, lps = [], [], [], []
            for k in range(K):
                if score[b, k] == -np.inf:
                    continue
                if fin[b, k]:
                    vals.append([score[b, k]]); par.append([k]); tok.append([eos]); lps.append([0.0])
                else:
                    vals.append(score[b, k] + logp[b, k]); par.append(np.full(V, k)); tok.append(np.arange(V)); lps.append(logp[b, k])
            vals, par, tok, lps = (np.concatenate(a) for a in (vals, par, tok, lps))
            keep = np.isfinite(vals)
            vals, par, tok, lps = vals[keep], par[keep], tok[keep], lps[keep]
            order = np.lexsort((tok, par, -vals))
            if len(order) > K:
                margins[b] = min(margins[b], float(vals[order[K - 1]] - vals[order[K]]))
            new_score = np.full(K, -np.inf, dtype=dtype)
            new_fin = np.ones(K, dtype=bool)
            new_hist_tok = np.full((K, S), eos, dtype=np.int64)
            new_hist_lp = np.zeros((K, S), dtype=dtype)
            for slot in range(K):
                if slot < len(order):
                    i = order[slot]
                    p = int(par[i])
                    new_score[slot], new_tok[b, slot], new_fin[slot] = vals[i], tok[i], tok[i] == eos
                    new_hist_tok[slot], new_hist_lp[slot] = hist_tok[b, p], hist_lp[b, p]
                    new_hist_tok[slot, s], new_hist_lp[slot, s] = tok[i], lps[i]
                else:
                    p = slot  # no finite candidate: the slot keeps its own state and scores -inf
                perm[b * K + slot] = b * K + p
            score[b], fin[b], hist_tok[b], hist_lp[b] = new_score, new_fin, new_hist_tok, new_hist_lp
        h = [x[perm] for x in h]
        c = [x[perm] for x in c]
        ctx = ctx[perm]
        word = np.eye(V, dtype=dtype)[new_tok.reshape(-1)]
    N = nbest
    tokens = np.full((B, N, S), eos, dtype=np.int64)
    token_logp = np.zeros((B, N, S), dtype=dtype)
    lengths = np.zeros((B, N), dtype=np.int64)
    scores = np.full((B, N), -np.inf, dtype=dtype)
    for b in range(B):
        length = np.zeros(K, dtype=np.int64)
        key = np.full(K, -np.inf, dtype=np.float32)
        for k in range(K):
            if score[b, k] == -np.inf:
                continue
            hit = np.nonzero(hist_tok[b, k] == eos)[0]
            length[k] = hit[0] + 1 if len(hit) else S
            key[k] = np.float32(score[b, k]) / np.power(np.float32(length[k]), np.float32(length_penalty))
        rank = np.argsort(-key, kind="stable")
        finite = key[rank[:N + 1]]
        finite = finite[np.isfinite(finite)]
        if len(finite) > 1:
            margins[b] = min(margins[b], float(np.min(finite[:-1] - finite[1:])))
        for n in range(N):
            k = rank[n]
            if score[b, k] == -np.inf:
                continue
            tokens[b, n], token_logp[b, n], lengths[b, n], scores[b, n] = hist_tok[b, k], hist_lp[b, k], length[k], score[b, k]
    return dict(tokens=tokens, token_logp=token_logp, lengths=lengths, scores=scores, margins=margins, min_margin=float(margins.min()))


def tiny_case(cfg="tiny", B=3, U=6, seed=4, gain=3.0):
    las = tl.build_model(cfg, max_label_len=4, seed=seed, gain=gain)
    c = tl.CONFIGS[cfg]
    enc = np.random.RandomState(seed).standard_normal((B, U, 2 * c["H"])) * 0.5
    return las, tl.state_dict_numpy(las), c, enc


@pytest.mark.parametrize("cfg", ["tiny", "tiny_gru", "tiny_mh"])
def test_width_one_is_greedy_decoding(cfg):
    las, sd, c, enc = tiny_case(cfg)
    S = 12
    g = O.speller_forward(enc, sd, c["sl"], S, dtype=np.float64)
    r = speller_beam_search(enc, sd, c["sl"], S, beam=1, nbest=1, eos=1)
    for b in range(enc.shape[0]):
        greedy = g["tokens"][:, b]
        hit = np.nonzero(greedy == 1)[0]
        n = hit[0] + 1 if len(hit) else S
        assert r["lengths"][b, 0] == n
        assert np.array_equal(r["tokens"][b, 0, :n], greedy[:n])
        assert np.all(r["tokens"][b, 0, n:] == 1) and np.all(r["token_logp"][b, 0, n:] == 0)
        lp = g["logp"][np.arange(n), b, greedy[:n]]
        assert np.array_equal(r["token_logp"][b, 0, :n], lp)
        assert r["scores"][b, 0] == pytest.approx(lp.sum(), abs=1e-12)


@pytest.mark.parametrize("alpha", [0.0, 0.7])
def test_wide_beam_over_two_steps_is_the_brute_force_n_best(alpha):
    """K >= V and S = 2: the hypotheses are (eos) and every (a, b) with a != eos; the beam keeps the K best by raw score and ranks
    those by score / length**alpha."""
    las, sd, c, enc = tiny_case("tiny", B=2)
    V, K, N = c["V"], 32, 32
    r = speller_beam_search(enc, sd, c["sl"], 2, beam=K, nbest=N, eos=1, length_penalty=alpha)
    lp0 = O.speller_forward(enc, sd, c["sl"], 1, dtype=np.float64)["logp"][0]
    for b in range(enc.shape[0]):
        hyps = [((1,), lp0[b, 1], 1)]
        for a in range(V):
            if a == 1:
                continue
            lp1 = O.speller_forward(enc[b:b + 1], sd, c["sl"], 2, ground_truth=np.array([[a, a]]), dtype=np.float64)["logp"][1, 0]
            hyps += [((a, v), lp0[b, a] + lp1[v], 2) for v in range(V)]
        hyps.sort(key=lambda t: -t[1])  # raw scores are distinct here
        kept = hyps[:K]
        keys = [np.float32(s) / np.power(np.float32(n), np.float32(alpha)) for _, s, n in kept]
        best = [kept[i] for i in np.argsort(-np.array(keys), kind="stable")[:N]]
        for n, (toks, s, length) in enumerate(best):
            assert tuple(r["tokens"][b, n, :length]) == toks and r["lengths"][b, n] == length
            assert r["scores"][b, n] == pytest.approx(s, abs=1e-12)


# ---- argument checks ------------------------------------------------------------------------------------------------------------

def _dims(**kw):
    d = dict(B=2, U=6, E=32, Hs=32, sl=2, V=30, D=16, heads=1, no_mlp=0, cell=0)
    d.update(kw)
    return _cabi.SpellerDims(*(d[k] for k, _ in _cabi.SpellerDims._fields_))


def _io(**kw):
    io = _cabi.BeamIO()
    io.enc, io.tokens, io.lengths, io.scores = 0x1000, 0x2000, 0x3000, 0x4000
    io.beam, io.nbest, io.eos_token, io.length_penalty = 4, 2, 1, 0.0
    for k, v in kw.items():
        setattr(io, k, v)
    return io


@pytest.mark.parametrize("field,value,msg", [
    ("beam", 0, b"beam width"), ("beam", 33, b"beam width"), ("nbest", 0, b"nbest"), ("nbest", 5, b"nbest"),
    ("eos_token", -1, b"eos_token"), ("eos_token", 30, b"eos_token"), ("length_penalty", -0.5, b"length_penalty"),
    ("length_penalty", math.inf, b"length_penalty"), ("length_penalty", math.nan, b"length_penalty"),
    ("enc", None, b"required"), ("tokens", None, b"required"), ("lengths", None, b"required"), ("scores", None, b"required"),
])
def test_beam_search_rejects_bad_arguments_before_touching_the_device(field, value, msg):
    lib = _cabi.load_library()
    d = _dims()
    st = lib.las_speller_beam_search(ctypes.byref(_io(**{field: value})), ctypes.c_void_p(0x5000), ctypes.byref(d), 8, 0, 1,
                                     ctypes.c_void_p(0x6000), 1 << 20, None)
    assert st == -1, st  # LAS_EINVAL
    assert msg in lib.las_last_error()


def test_beam_search_rejects_null_buffers_and_bad_steps():
    lib = _cabi.load_library()
    d = _dims()
    for packed, ws, steps, msg in ((None, 0x6000, 8, b"null pointer"), (0x5000, None, 8, b"null pointer"), (0x5000, 0x6000, 0, b"steps")):
        st = lib.las_speller_beam_search(ctypes.byref(_io()), packed, ctypes.byref(d), steps, 0, 1, ws, 1 << 20, None)
        assert st == -1 and msg in lib.las_last_error(), (packed, ws, steps)
    assert lib.las_speller_beam_search(None, 0x5000, ctypes.byref(d), 8, 0, 1, 0x6000, 1 << 20, None) == -1
    # valid arguments get past the checks: without a device the call fails there, not with LAS_EINVAL
    if not torch.cuda.is_available():
        assert lib.las_speller_beam_search(ctypes.byref(_io()), 0x5000, ctypes.byref(d), 8, 0, 1, 0x6000, 1 << 20, None) != -1


def test_beam_size_queries():
    lib = _cabi.load_library()
    d = _dims()
    for mode in (_cabi.MODE_FP32, _cabi.MODE_BF16):
        ws = lib.las_speller_beam_workspace_bytes(ctypes.byref(d), 10, 4, mode)
        assert ws >= 4 * (2 * 4 * (30 + 32) + 3 * 2 * 2 * 4 * 32 + 3 * 10 * 2 * 4)
        assert lib.las_speller_beam_workspace_bytes(ctypes.byref(d), 10, 8, mode) > ws
        assert lib.las_speller_beam_packed_bytes(ctypes.byref(d), mode) >= lib.las_speller_packed_bytes(ctypes.byref(d), _cabi.MODE_FP32)
    for steps, beam in ((0, 4), (-1, 4), (10, 0), (10, 33)):
        assert lib.las_speller_beam_workspace_bytes(ctypes.byref(d), steps, beam, 0) == 0, (steps, beam)
    assert lib.las_speller_beam_workspace_bytes(ctypes.byref(d), 10, 4, 7) == 0
    bad = _dims(Hs=48)  # Hs != E
    assert lib.las_speller_beam_packed_bytes(ctypes.byref(bad), 0) == 0
    assert lib.las_speller_beam_workspace_bytes(ctypes.byref(bad), 10, 4, 0) == 0
    # fp32 mode: the beam pack is the ordinary pack; the tensor-core modes always carry the generic layout
    paper = _dims(B=8, U=100, E=512, Hs=512, D=64)
    assert lib.las_speller_beam_packed_bytes(ctypes.byref(paper), 0) == lib.las_speller_packed_bytes(ctypes.byref(paper), 0)
    assert lib.las_speller_beam_packed_bytes(ctypes.byref(paper), 1) > lib.las_speller_packed_bytes(ctypes.byref(paper), 0)


@pytest.mark.parametrize("kw", [dict(beam_width=0), dict(beam_width=33), dict(beam_width=2.0), dict(nbest=0), dict(beam_width=2, nbest=3),
                                dict(length_penalty=-1.0), dict(length_penalty=float("nan")), dict(length_penalty=float("inf")),
                                dict(max_steps=0)])
def test_python_beam_search_raises_value_error_on_the_host(kw):
    las = tl.build_model("tiny", max_label_len=6)
    enc = torch.zeros(2, 4, 32)  # on the CPU: the check must come before the device is needed
    with pytest.raises(ValueError):
        las.speller.beam_search(enc, **kw)
    if "max_steps" not in kw:
        with pytest.raises(ValueError):
            las.beam_search(torch.zeros(2, 16, 40), **kw)


def test_python_beam_search_checks_shapes_and_eos():
    las = tl.build_model("tiny", max_label_len=6)
    with pytest.raises(ValueError):
        las.speller.beam_search(torch.zeros(2, 4, 48))
    with pytest.raises(ValueError):
        las.speller.beam_search(torch.zeros(2, 4, 32), enc_lengths=torch.ones(3, dtype=torch.int32))
    las.speller.eos_token = 30
    with pytest.raises(ValueError):
        las.speller.beam_search(torch.zeros(2, 4, 32))
    las.speller.eos_token = 1
    with pytest.raises(RuntimeError, match="no CPU fallback"):  # valid arguments: the missing device is the next thing reported
        las.speller.beam_search(torch.zeros(2, 4, 32))
