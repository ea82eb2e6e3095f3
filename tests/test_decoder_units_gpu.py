"""The persistent decoder's LSTM CTAs in their two widths, and the serving pipeline's two schedules.

A CTA owns 16 hidden units (64 gate rows) or 32 (128 gate rows: every lane of its M = 128 MMAs); las_debug_set_option(30, .) forces
one (by default only the decoder launch the serving pipeline runs beside the next batch's listener takes 32).  The 32-unit CTA
builds its atoms from the same packed image and every output column is the same sum of the same products, so both widths must give
the same outputs bit for bit.

The serving pipeline runs the next batch's listener beside one decoder launch where the decoder leaves room for it, and around
decoder segments otherwise (las_debug_set_option(31, 0) forces the segmented schedule); both must give what LAS.forward gives.
"""
import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi

pytestmark = pytest.mark.gpu

HS16 = dict(F=40, H=8, L=2, sl=2, V=30, D=16)  # speller hidden size 16: one 16-unit block, a half-empty 32-unit CTA


def _bf16_or_skip():
    if not _cabi.load_library().las_mode_available(_cabi.MODE_BF16):
        pytest.skip("bf16 mode not built")


class _Option:
    def __init__(self, key, value, default):
        self.key, self.value, self.default = key, value, default

    def __enter__(self):
        assert _cabi.load_library().las_debug_set_option(self.key, self.value) == 0

    def __exit__(self, *exc):
        assert _cabi.load_library().las_debug_set_option(self.key, self.default) == 0


def _decode(las, enc, steps, **kw):
    logp, attn, tok = las.speller._decode(enc, steps, **kw)
    torch.cuda.synchronize()
    return logp.clone(), attn.clone(), tok.clone()


@pytest.mark.parametrize("cfg,B,T,S", [("paper", 64, 320, 40), ("paper", 32, 320, 40), ("paper", 17, 160, 24), ("small", 5, 64, 30),
                                       ("odd", 20, 96, 24), (HS16, 7, 64, 20)], ids=["paper64", "paper32", "paper17", "small5", "odd20", "hs16"])
def test_32_unit_ctas_equal_16_unit_ctas(cfg, B, T, S):
    """Key 30 = 16 against 32: logp, attention and tokens bit for bit in every feedback mode (greedy, raw, sampling, index and dense
    teacher forcing, the fused loss), with length masks and segmented, in two utterance groups (B = 64) and in one -- including the
    odd model (Hs = 48: the second 32-unit CTA of each layer has 16 units past Hs) and Hs = 16 (one CTA per layer, half of it empty)."""
    _bf16_or_skip()
    c = tl.CONFIGS[cfg] if isinstance(cfg, str) else cfg
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=29)
    for dm in (1, 0, 2):
        las = tl.build_model(cfg, max_label_len=S, decode_mode=dm, seed=29, gain=3.0, precision="bf16").cuda()
        enc = las.listener(x.cuda())
        U = enc.shape[1]
        lens = torch.tensor([U - (i % 5) for i in range(B)], dtype=torch.int32, device="cuda")
        variants = [dict(), dict(enc_lengths=lens), dict(segment_steps=10)]
        if dm == 1:
            variants += [dict(gt_index=labels.cuda().to(torch.int32).contiguous()),
                         dict(gt_dense=tl.onehot(labels, c["V"]).float().cuda().contiguous()),
                         dict(nll_labels=labels.cuda())]
        for kw in variants:
            outs = []
            for units in (16, 32):
                with _Option(30, units, 0):
                    torch.manual_seed(5)
                    outs.append(_decode(las, enc, S, **kw))
            for a, b in zip(*outs):
                assert torch.equal(a, b), (cfg, B, dm, list(kw))


def test_32_units_in_lockstep_are_refused():
    """32-unit CTAs serve at most 32 rows per iteration: forcing them on 64 utterances in lockstep is an error, not a wrong result."""
    _bf16_or_skip()
    c = tl.CONFIGS["tiny"]
    las = tl.build_model("tiny", max_label_len=4, seed=3, precision="bf16").cuda()
    x, _ = tl.make_inputs(64, 32, c["F"], 4, c["V"], seed=3)
    enc = las.listener(x.cuda())
    with _Option(19, 0, 1), _Option(30, 32, 0):
        with pytest.raises(Exception, match="32 rows per iteration"):
            _decode(las, enc, 4)


@pytest.mark.parametrize("cfgname,B,T,S", [("paper", 64, 1600, 300), ("paper", 16, 3000, 600), ("odd", 3, 48, 6)],
                         ids=["c3", "c4", "odd"])
def test_serving_schedules_equal_forward(cfgname, B, T, S):
    """LAS.serve() under the beside schedule (key 31 = 1, the default) and the segmented one (key 31 = 0): every batch gets exactly
    what LAS.forward gives it, over two rounds (the pipeline's workspaces and events are reused)."""
    _bf16_or_skip()
    c = tl.CONFIGS[cfgname]
    las = tl.build_model(cfgname, max_label_len=S, seed=17, gain=3.0, precision="bf16").cuda()
    xs = [tl.make_inputs(B, T, c["F"], S, c["V"], seed=200 + i)[0].cuda() for i in range(3)]
    want = []
    for x in xs:
        preds, attns = las(x, None, 0.0, is_training=False)
        want.append((torch.stack(preds).clone(), torch.stack([a[0] for a in attns]).clone(), las.speller.last_tokens.clone()))
    for beside in (1, 0):
        with _Option(31, beside, 1):
            for _ in range(2):
                pipe = las.serve()
                got = [r for r in (pipe.submit(x) for x in xs) if r is not None]
                got.append(pipe.flush())
                torch.cuda.synchronize()
                assert len(got) == len(xs)
                for (lp, at, tk), r in zip(want, got):
                    assert torch.equal(r.tokens, tk), (cfgname, beside)
                    assert torch.equal(r.logp, lp), (cfgname, beside)
                    assert torch.equal(r.attn, at), (cfgname, beside)
