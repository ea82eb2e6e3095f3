"""numpy restatement of the LAS forward hot path (TEST INFRASTRUCTURE -- see oracle/__init__.py).

Follows, function by function, jiwidi/las-pytorch:
  * pyramid fold            model/las_model.py:82-87
  * BLSTM layer             model/las_model.py:72-79,90   (torch nn.LSTM equations, gate order i,f,g,o,
                                                            zero initial state, reverse direction walks t downwards)
  * Listener stack          model/las_model.py:116-134
  * psi / phi / attention   model/las_model.py:276-297 + utils/functions.py:72-77 (TimeDistributed)
  * Speller step + loop     model/las_model.py:178-184, 186-238 + utils/functions.py:54-63 (<sos> one-hot)
  * LAS.forward dispatch    model/las_model.py:30-40

The arithmetic of those call sites lives in torch (requirements.txt:5 pins torch==1.5.0; this image has
2.11.0).  It is restated here from torch's documented LSTM / Linear / softmax definitions.

Parity pin: checked against outputs of the reference itself (tests/golden/*.npz, produced by
tests/golden/make_golden.py from the unmodified /root/reference code) by tests/test_oracle_golden.py.

Weights are passed as a dict {state_dict key -> ndarray} using the reference's own key names
(SURVEY.md A.2), so a reference checkpoint's `package["state_dict"]` can be fed in unchanged.
All functions run in the dtype of `dtype` (np.float32 or np.float64).
"""
from __future__ import annotations

import numpy as np


def _sigmoid(x):
    return 1.0 / (1.0 + np.exp(-x))


def _w(sd, key, dtype):
    return np.asarray(sd[key], dtype=dtype)


def pyramid_fold(x):
    """[B, T, F] -> [B, T//2, 2F]; row t = frame 2t || frame 2t+1.  model/las_model.py:82-87.

    The reference does `view(B, int(T/2), 2F)`, which raises for odd T; so do we.
    """
    b, t, f = x.shape
    if t % 2:
        raise RuntimeError(f"shape '[{b}, {t // 2}, {2 * f}]' is invalid for input of size {b * t * f}")
    return np.ascontiguousarray(x).reshape(b, t // 2, 2 * f)


def lstm_cell(pre, c):
    """One LSTM cell update from gate pre-activations `pre` [B,4H] (order i,f,g,o) and cell state c [B,H]."""
    hdim = c.shape[1]
    i = _sigmoid(pre[:, 0 * hdim:1 * hdim])
    f = _sigmoid(pre[:, 1 * hdim:2 * hdim])
    g = np.tanh(pre[:, 2 * hdim:3 * hdim])
    o = _sigmoid(pre[:, 3 * hdim:4 * hdim])
    c_new = f * c + i * g
    h_new = o * np.tanh(c_new)
    return h_new, c_new


def rnn_cell_step(px, ph, h, c):
    """One step of the cell the weights describe -- torch nn.LSTM / nn.GRU / nn.RNN equations.  px = x . W_ih^T + b_ih,
    ph = h . W_hh^T + b_hh, both [B, G*H]; G = 4: LSTM (i,f,g,o), 3: GRU (r,z,n), 1: RNN (tanh).  The reference builds the
    module with getattr(nn, rnn_unit.upper()) (model/las_model.py:69,156)."""
    hdim = h.shape[1]
    gates = px.shape[1] // hdim
    if gates == 4:
        return lstm_cell(px + ph, c)
    if gates == 3:
        r = _sigmoid(px[:, :hdim] + ph[:, :hdim])
        z = _sigmoid(px[:, hdim:2 * hdim] + ph[:, hdim:2 * hdim])
        n = np.tanh(px[:, 2 * hdim:] + r * ph[:, 2 * hdim:])
        return (1 - z) * n + z * h, c
    return np.tanh(px + ph), c


def lstm_direction(xr, w_ih, w_hh, b_ih, b_hh, reverse):
    """One direction of a 1-layer nn.LSTM / nn.GRU / nn.RNN(batch_first=True) over xr [B,Tl,K] -> [B,Tl,H]."""
    b, tl, _ = xr.shape
    hdim = w_hh.shape[1]
    # input projection for all timesteps at once (SURVEY.md row a3)
    p = xr.reshape(b * tl, -1) @ w_ih.T + b_ih
    p = p.reshape(b, tl, -1)
    h = np.zeros((b, hdim), dtype=xr.dtype)
    c = np.zeros((b, hdim), dtype=xr.dtype)
    out = np.empty((b, tl, hdim), dtype=xr.dtype)
    steps = range(tl - 1, -1, -1) if reverse else range(tl)
    for t in steps:  # recurrence (row a4)
        h, c = rnn_cell_step(p[:, t], h @ w_hh.T + b_hh, h, c)
        out[:, t] = h
    return out


def pblstm_layer(x, sd, prefix, dtype):
    """model/las_model.py:81-91 -- fold time, then bidirectional LSTM; output [fwd H || bwd H]."""
    xr = pyramid_fold(x)
    outs = []
    for sfx, rev in (("", False), ("_reverse", True)):
        outs.append(
            lstm_direction(
                xr,
                _w(sd, f"{prefix}.BLSTM.weight_ih_l0{sfx}", dtype),
                _w(sd, f"{prefix}.BLSTM.weight_hh_l0{sfx}", dtype),
                _w(sd, f"{prefix}.BLSTM.bias_ih_l0{sfx}", dtype),
                _w(sd, f"{prefix}.BLSTM.bias_hh_l0{sfx}", dtype),
                rev,
            )
        )
    return np.concatenate(outs, axis=-1)


def listener_forward(x, sd, num_layers, dtype=np.float32, prefix="listener"):
    """model/las_model.py:129-134 -- chain pLSTM_layer0..L-1; [B,T,F] -> [B,T/2^L,2H]."""
    out = np.asarray(x, dtype=dtype)
    for layer in range(num_layers):
        out = pblstm_layer(out, sd, f"{prefix}.pLSTM_layer{layer}", dtype)
    return out


def listener_forward_masked(x, lengths, sd, num_layers, dtype=np.float32, prefix="listener"):
    """Length-mask EXTENSION (not in the reference, which runs over the zero padding -- SURVEY.md A.5.2; the lengths are
    the `inputs_length` that utils/data.py:146 computes and train.py:117 drops).  Layer l keeps len_l = ceil(len_{l-1}/2)
    steps; each direction runs over the valid prefix only and outputs past it are zero -- the semantics of torch's
    pack_padded_sequence -> nn.LSTM -> pad_packed_sequence, which tests/test_oracle_golden.py pins this function to.
    Returns (enc [B,U,2H], enc_lengths [B])."""
    out = np.asarray(x, dtype=dtype)
    lens = np.asarray(lengths, dtype=np.int64)
    for layer in range(num_layers):
        xr = pyramid_fold(out)
        lens = np.minimum((lens + 1) // 2, xr.shape[1])
        nxt = np.zeros((xr.shape[0], xr.shape[1], 2 * sd[f"{prefix}.pLSTM_layer{layer}.BLSTM.weight_hh_l0"].shape[1]), dtype=dtype)
        for b in range(xr.shape[0]):
            n = int(lens[b])
            if n > 0:  # utterance b alone, truncated to its valid steps
                nxt[b, :n] = pblstm_layer(out[b:b + 1, :2 * n], sd, f"{prefix}.pLSTM_layer{layer}", dtype)[0]
        out = nxt
    return out, lens


def psi_project(enc, sd, dtype=np.float32, prefix="speller", activate=True):
    """relu(TimeDistributed(psi, enc)) -- model/las_model.py:279 + utils/functions.py:72-77.

    Step-invariant, so computed once (the reference recomputes identical values every step)."""
    b, u, e = enc.shape
    k = enc.reshape(b * u, e) @ _w(sd, f"{prefix}.attention.psi.weight", dtype).T
    k = k + _w(sd, f"{prefix}.attention.psi.bias", dtype)
    if activate:
        k = np.maximum(k, 0)
    return k.reshape(b, u, -1)


def _attend_one(q, enc, keys, enc_lengths):
    energy = np.einsum("bd,bud->bu", q, keys)
    if enc_lengths is not None:
        mask = np.arange(enc.shape[1])[None, :] >= np.asarray(enc_lengths)[:, None]
        energy = np.where(mask, -np.inf, energy)
    energy = energy - energy.max(axis=-1, keepdims=True)
    w = np.exp(energy)
    score = w / w.sum(axis=-1, keepdims=True)
    return score, np.einsum("bu,bue->be", score, enc)


def attention(state, enc, psi, sd, dtype=np.float32, prefix="speller", activate=True, enc_lengths=None):
    """'dot' attention -- model/las_model.py:275-314.

    state [B,Hs], enc [B,U,E], psi [B,U,D] -> (score [B,U] or list of per-head scores, context [B,E]).
    Variants, selected by the keys present in `sd` exactly as the reference module is built (:264-273):
      * no `attention.phi.weight`  -> use_mlp_in_attention=False (:283-285): query = state, keys = enc;
      * `attention.dim_reduce.weight` present -> multi_head > 1 (:298-314): phi's output is split into heads of D
        columns, every head attends over the same keys, the contexts are concatenated and reduced.
    `enc_lengths` (None in the reference) masks encoder steps >= length before the softmax."""
    if f"{prefix}.attention.phi.weight" not in sd:
        score, context = _attend_one(state, enc, enc, enc_lengths)
        return score.astype(dtype), context.astype(dtype)
    q = state @ _w(sd, f"{prefix}.attention.phi.weight", dtype).T + _w(sd, f"{prefix}.attention.phi.bias", dtype)
    if activate:
        q = np.maximum(q, 0)
    if f"{prefix}.attention.dim_reduce.weight" not in sd:
        score, context = _attend_one(q, enc, psi, enc_lengths)
        return score.astype(dtype), context.astype(dtype)
    d = psi.shape[-1]
    scores, ctxs = [], []
    for hd in range(q.shape[1] // d):
        s_h, c_h = _attend_one(q[:, hd * d:(hd + 1) * d], enc, psi, enc_lengths)
        scores.append(s_h.astype(dtype))
        ctxs.append(c_h)
    context = np.concatenate(ctxs, axis=-1) @ _w(sd, f"{prefix}.attention.dim_reduce.weight", dtype).T
    context = context + _w(sd, f"{prefix}.attention.dim_reduce.bias", dtype)
    return scores, context.astype(dtype)


def log_softmax(z):
    z = z - z.max(axis=-1, keepdims=True)
    return z - np.log(np.exp(z).sum(axis=-1, keepdims=True))


def speller_forward(
    enc,
    sd,
    num_layers,
    steps,
    ground_truth=None,
    decode_mode=1,
    dtype=np.float32,
    prefix="speller",
    enc_lengths=None,
    activate=True,
):
    """Speller step loop -- model/las_model.py:186-238 with forward_step :178-184.

    enc          [B,U,E] listener features
    ground_truth None (free running) or int array [B,S] of label indices / one-hot [B,S,V]
                 (teacher forcing: next input is ground_truth[:, step], NOT shifted -- :216-217)
    steps        number of decode steps (max_label_len free-running, ground_truth.shape[1] teacher-forced)
    decode_mode  0: feed log-probs back (:220-221); 1: one-hot(argmax) (:223-227)
    activate     relu on phi(state) and psi(enc) (mlp_activate_in_attention="relu"); False: both used raw ("None")
    returns dict(logp [S,B,V], attn [S,B,U], tokens [S,B] argmax of logp, context [S,B,E])
    """
    enc = np.asarray(enc, dtype=dtype)
    b, u, e = enc.shape
    w_cd = _w(sd, f"{prefix}.character_distribution.weight", dtype)
    b_cd = _w(sd, f"{prefix}.character_distribution.bias", dtype)
    v = w_cd.shape[0]
    hs = _w(sd, f"{prefix}.rnn_layer.weight_hh_l0", dtype).shape[1]
    if ground_truth is not None:
        gt = np.asarray(ground_truth)
        if gt.ndim == 2:
            gt = np.eye(v, dtype=dtype)[gt]
        gt = gt.astype(dtype)

    psi = psi_project(enc, sd, dtype, prefix, activate) if f"{prefix}.attention.psi.weight" in sd else enc
    h = [np.zeros((b, hs), dtype=dtype) for _ in range(num_layers)]  # hidden_state=None -> zeros
    c = [np.zeros((b, hs), dtype=dtype) for _ in range(num_layers)]
    word = np.zeros((b, v), dtype=dtype)
    word[:, 0] = 1  # <sos> = index 0 (:193-195)
    ctx = enc[:, 0, :]  # first "context" is encoder frame 0 (:198)

    logps, attns, toks, ctxs = [], [], [], []
    for s in range(steps):
        inp = np.concatenate([word, ctx], axis=-1)  # [B, V+E] (:198,:236)
        for l in range(num_layers):  # stacked cells, seq-len 1 (:179)
            px = inp @ _w(sd, f"{prefix}.rnn_layer.weight_ih_l{l}", dtype).T + _w(sd, f"{prefix}.rnn_layer.bias_ih_l{l}", dtype)
            ph = h[l] @ _w(sd, f"{prefix}.rnn_layer.weight_hh_l{l}", dtype).T + _w(sd, f"{prefix}.rnn_layer.bias_hh_l{l}", dtype)
            h[l], c[l] = rnn_cell_step(px, ph, h[l], c[l])
            inp = h[l]
        score, ctx = attention(h[-1], enc, psi, sd, dtype, prefix, activate, enc_lengths)  # (:180)
        logp = log_softmax(np.concatenate([h[-1], ctx], axis=-1) @ w_cd.T + b_cd)  # (:181-182)
        tok = logp.argmax(axis=-1)
        logps.append(logp.astype(dtype))
        attns.append(score)
        toks.append(tok)
        ctxs.append(ctx)
        if ground_truth is not None:
            word = gt[:, s, :]
        elif decode_mode == 0:
            word = logp
        else:
            word = np.eye(v, dtype=dtype)[tok]
    return {
        "logp": np.stack(logps),
        "attn": np.stack(attns),
        "tokens": np.stack(toks).astype(np.int64),
        "context": np.stack(ctxs),
    }


def las_forward(
    x,
    sd,
    listener_layers,
    speller_layers,
    max_label_len,
    ground_truth=None,
    teacher_forced=False,
    decode_mode=1,
    dtype=np.float32,
    activate=True,
):
    """LAS.forward -- model/las_model.py:30-40.  The teacher-forcing coin flip (:189) is resolved by the
    caller (`teacher_forced`), which also fixes the step count (:205-208)."""
    enc = listener_forward(x, sd, listener_layers, dtype)
    if teacher_forced and ground_truth is not None:
        steps = np.asarray(ground_truth).shape[1]
        out = speller_forward(enc, sd, speller_layers, steps, ground_truth, decode_mode, dtype, activate=activate)
    else:
        out = speller_forward(enc, sd, speller_layers, max_label_len, None, decode_mode, dtype, activate=activate)
    out["enc"] = enc
    return out


# ---- solver epilogue ("next" row f1): solver/solver.py:11-24, 33-45, 70-92 --------------------------------

def levenshtein(a, b):
    """editdistance.eval stand-in (the `editdistance` package is not in this image)."""
    prev = list(range(len(b) + 1))
    for i, ca in enumerate(a, 1):
        cur = [i]
        for j, cb in enumerate(b, 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (ca != cb)))
        prev = cur
    return prev[-1]


def letter_error_rate(pred_tokens, true_tokens):
    """solver/solver.py:11-24.  pred cut at first <eos>=1, zeros dropped; truth drops 0 and 1."""
    out = []
    for p, t in zip(pred_tokens, true_tokens):
        ct = [int(w) for w in t if (w != 1 and w != 0)]
        cp = []
        for w in p:
            if w == 0:
                continue
            if w == 1:
                break
            cp.append(int(w))
        out.append(levenshtein(cp, ct) / len(ct))
    return out


def nll_loss_ignore0(logp_bsv, label_idx):
    """solver/solver.py:62,70-77 -- NLLLoss(ignore_index=0) averaged over non-ignored targets."""
    b, s, v = logp_bsv.shape
    flat = logp_bsv.reshape(b * s, v)
    idx = np.asarray(label_idx).reshape(-1)
    keep = idx != 0
    picked = flat[np.arange(b * s), idx]
    return float(-(picked[keep]).sum() / max(int(keep.sum()), 1))


def label_smoothing_loss(logp_bsv, onehot_bsv, label_smoothing=0.1):
    """solver/solver.py:33-45."""
    true_y = np.asarray(onehot_bsv, dtype=logp_bsv.dtype)
    seq_len = true_y.sum(-1).sum(-1, keepdims=True)
    class_dim = true_y.shape[-1]
    smooth = ((1.0 - label_smoothing) * true_y + (label_smoothing / class_dim)) * true_y.sum(-1, keepdims=True)
    return float(-np.mean(((smooth * logp_bsv).sum(-1) / seq_len).sum(-1)))

