"""The fp64 oracle's attention without an activation (mlp_activate_in_attention="None") against an independent torch restatement of the
reference's Attention.forward (model/las_model.py:275-314) and Speller step (:178-184): with no activation, phi(state) and psi(enc) are
used raw.  The GPU tests of that setting (tests/test_decoder_variants_gpu.py) take the oracle as ground truth."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import las_testlib as tl
from oracle import las_oracle as O


def model_sd(heads=1, sl=2):
    cfg = dict(F=40, H=16, L=1, sl=sl, V=30, D=8, heads=heads, activate="None")
    las = tl.build_model(cfg, max_label_len=3, seed=7, gain=2.5)
    assert las.speller.attention.activate is None and las.speller.attention.relu_flag == 0
    return cfg, {k: torch.from_numpy(v).double() for k, v in tl.state_dict_numpy(las).items()}


def torch_attention(state, enc, sd, heads):
    """Attention.forward with activate=None: energies <phi(state), psi(enc)> per head, softmax, context; heads > 1 concatenate their
    contexts and reduce them with dim_reduce."""
    q = F.linear(state, sd["speller.attention.phi.weight"], sd["speller.attention.phi.bias"])
    k = F.linear(enc, sd["speller.attention.psi.weight"], sd["speller.attention.psi.bias"])
    d = k.shape[-1]
    scores, ctxs = [], []
    for h in range(heads):
        energy = torch.bmm(k, q[:, h * d:(h + 1) * d].unsqueeze(2)).squeeze(2)
        score = torch.softmax(energy, dim=-1)
        scores.append(score)
        ctxs.append(torch.bmm(score.unsqueeze(1), enc).squeeze(1))
    if heads == 1:
        return scores[0], ctxs[0]
    return scores, F.linear(torch.cat(ctxs, dim=-1), sd["speller.attention.dim_reduce.weight"], sd["speller.attention.dim_reduce.bias"])


@pytest.mark.parametrize("heads", [1, 3])
def test_attention_without_activation_matches_a_torch_restatement(heads):
    cfg, sd = model_sd(heads)
    g = torch.Generator().manual_seed(3)
    enc = torch.randn(4, 9, 2 * cfg["H"], generator=g, dtype=torch.float64)
    state = torch.randn(4, 2 * cfg["H"], generator=g, dtype=torch.float64)
    want_s, want_c = torch_attention(state, enc, sd, heads)
    sdn = {k: v.numpy() for k, v in sd.items()}
    psi = O.psi_project(enc.numpy(), sdn, np.float64, activate=False)
    got_s, got_c = O.attention(state.numpy(), enc.numpy(), psi, sdn, np.float64, activate=False)
    for gs, ws in zip(got_s if heads > 1 else [got_s], want_s if heads > 1 else [want_s]):
        assert np.abs(gs - ws.numpy()).max() <= 1e-12
    assert np.abs(got_c - want_c.numpy()).max() <= 1e-12
    # the activation is not a no-op here: relu moves the result
    relu_s, _ = O.attention(state.numpy(), enc.numpy(), O.psi_project(enc.numpy(), sdn, np.float64), sdn, np.float64)
    assert np.abs(np.asarray(relu_s) - np.asarray(got_s)).max() > 1e-3


def test_speller_forward_without_activation_matches_a_torch_restatement():
    cfg, sd = model_sd()
    B, U, S, V, sl = 3, 7, 3, cfg["V"], cfg["sl"]
    g = torch.Generator().manual_seed(5)
    enc = torch.tanh(torch.randn(B, U, 2 * cfg["H"], generator=g, dtype=torch.float64))
    labels = torch.randint(2, V, (B, S), generator=g)
    # the reference's step loop (:186-238), teacher forced with the labels, LSTM cells in gate order i, f, g, o
    hs = 2 * cfg["H"]
    h = [torch.zeros(B, hs, dtype=torch.float64) for _ in range(sl)]
    c = [torch.zeros(B, hs, dtype=torch.float64) for _ in range(sl)]
    word = F.one_hot(torch.zeros(B, dtype=torch.int64), V).double()
    ctx = enc[:, 0]
    want_lp, want_at = [], []
    for s in range(S):
        x = torch.cat([word, ctx], dim=-1)
        for layer in range(sl):
            gates = F.linear(x, sd[f"speller.rnn_layer.weight_ih_l{layer}"], sd[f"speller.rnn_layer.bias_ih_l{layer}"]) + \
                F.linear(h[layer], sd[f"speller.rnn_layer.weight_hh_l{layer}"], sd[f"speller.rnn_layer.bias_hh_l{layer}"])
            i, f, gg, o = gates.chunk(4, dim=-1)
            c[layer] = torch.sigmoid(f) * c[layer] + torch.sigmoid(i) * torch.tanh(gg)
            h[layer] = torch.sigmoid(o) * torch.tanh(c[layer])
            x = h[layer]
        score, ctx = torch_attention(h[-1], enc, sd, 1)
        logits = F.linear(torch.cat([h[-1], ctx], dim=-1), sd["speller.character_distribution.weight"], sd["speller.character_distribution.bias"])
        want_lp.append(F.log_softmax(logits, dim=-1))
        want_at.append(score)
        word = F.one_hot(labels[:, s], V).double()
    sdn = {k: v.numpy() for k, v in sd.items()}
    got = O.speller_forward(enc.numpy(), sdn, sl, S, ground_truth=labels.numpy(), dtype=np.float64, activate=False)
    assert np.abs(got["logp"] - torch.stack(want_lp).numpy()).max() <= 1e-12
    assert np.abs(got["attn"] - torch.stack(want_at).numpy()).max() <= 1e-12
    relu = O.speller_forward(enc.numpy(), sdn, sl, S, ground_truth=labels.numpy(), dtype=np.float64)
    assert np.abs(relu["attn"] - got["attn"]).max() > 1e-3
