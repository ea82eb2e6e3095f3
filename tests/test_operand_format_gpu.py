"""bf16 and fp16 models used one after the other on one host thread.  The 16-bit operand format of every pack, GEMM and decoder launch
follows the mode of its own call, so interleaving calls of the two modes changes none of their outputs."""
import ctypes as C

import numpy as np
import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi

pytestmark = pytest.mark.gpu

B, T, S = 4, 128, 16


def outputs(las, kind, x, x2, labels):
    """One call of `kind` on `las`, its outputs on the host; the first one is a float tensor (log-probs or scores)."""
    if kind == "teacher_forced":
        np.random.seed(0)
        preds, attns = las(x, labels, 1.1, is_training=True)
        return [torch.stack(preds).cpu(), torch.stack([a[0] for a in attns]).cpu()]
    if kind == "greedy":
        np.random.seed(0)
        preds, attns = las(x, None, 0.0, is_training=False)
        return [torch.stack(preds).cpu(), torch.stack([a[0] for a in attns]).cpu(), las.speller.last_tokens.cpu()]
    if kind == "serve":  # the second submit decodes x while it encodes x2 (las_pipeline_step)
        pipe = las.serve()
        assert pipe.submit(x) is None
        r1 = pipe.submit(x2)
        r2 = pipe.flush()
        return [t.cpu() for r in (r1, r2) for t in (r.logp, r.attn, r.tokens)]
    r = las.beam_search(x, beam_width=4, nbest=2)
    return [r.scores.cpu(), r.token_logp.cpu(), r.tokens.cpu(), r.lengths.cpu()]


@pytest.mark.parametrize("cfg", ["paper", "tiny_gru"])
def test_interleaved_precisions_compute_what_each_computes_alone(cfg):
    """paper: the cluster-resident listener, the persistent decoder and the concurrent serving step, with beam search on the generic
    step; tiny_gru: the generic tensor-core listener and the fused generic decoder step."""
    lib = _cabi.load_library()
    assert lib.las_mode_available(_cabi.MODE_BF16) and lib.las_mode_available(_cabi.MODE_F16)
    c = tl.CONFIGS[cfg]
    x, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=5)
    x2, _ = tl.make_inputs(B, T, c["F"], S, c["V"], seed=6)
    x, x2, labels = x.cuda(), x2.cuda(), tl.onehot(labels, c["V"]).cuda()
    models = {p: tl.build_model(cfg, max_label_len=S, seed=17, gain=3.0, precision=p).cuda() for p in ("bf16", "fp16")}
    if cfg == "paper":
        ld = _cabi.ListenerDims(B, T, c["F"], c["H"], c["L"], 0)
        sd = models["bf16"].speller._dims(B, T >> c["L"], 2 * c["H"])
        for mode in (_cabi.MODE_BF16, _cabi.MODE_F16):
            assert lib.las_pipeline_overlaps(C.byref(ld), C.byref(sd), S, mode) == 1
    kinds = ["teacher_forced", "greedy", "serve", "beam"]

    alone = {(p, k): outputs(models[p], k, x, x2, labels) for p in ("bf16", "fp16") for k in kinds}
    for k in kinds:
        assert not torch.equal(alone[("bf16", k)][0], alone[("fp16", k)][0]), f"{k}: bf16 and fp16 give the same bits"

    # again with the precision switching at every call, packing included
    for las in models.values():
        las.invalidate_packed_weights()
    order = [("bf16", "teacher_forced"), ("fp16", "teacher_forced"), ("bf16", "greedy"), ("fp16", "greedy"),
             ("bf16", "serve"), ("fp16", "beam"), ("bf16", "beam"), ("fp16", "serve")]
    for p, k in order:
        got = outputs(models[p], k, x, x2, labels)
        want = alone[(p, k)]
        assert len(got) == len(want)
        for i, (g, w) in enumerate(zip(got, want)):
            assert torch.equal(g, w), f"{p} {k}: output {i} differs from the same call made alone"
