"""Byte counts of the packed-weight and workspace layouts, and the argument checks of las_pipeline_step, on the host.

Callers allocate packs and workspaces from the six size queries, so their values are part of the ABI.  The table in
tests/golden/layout_sizes.json pins them for every mode and model variant.  The queries need no device: without one,
sm_count() assumes the B200's 148 SMs, and the SM count decides whether the persistent decoder covers a shape.  Rewrite
the table (`python tests/test_layout_sizes_cpu.py > tests/golden/layout_sizes.json`) only with a deliberate layout change.
"""
import ctypes
import json
import os
import sys

import pytest

import las_testlib as tl
from las_pytorch_b200 import _cabi

TABLE = os.path.join(tl.GOLDEN_DIR, "layout_sizes.json")

# name -> (model config, listener input frames T); the encoder has U = T / 2^L steps
CONFIGS = {
    "tiny": (tl.CONFIGS["tiny"], 64),
    "odd": (tl.CONFIGS["odd"], 96),
    "small": (tl.CONFIGS["small"], 1600),
    "paper": (tl.CONFIGS["paper"], 1600),
    "shipped": (tl.CONFIGS["shipped"], 1600),  # config/librispeech-config.yaml: speller 1024 x 2
    "gru": (tl.CONFIGS["tiny_gru"], 64),
    "rnn": (tl.CONFIGS["tiny_rnn"], 64),
    "multi_head": (tl.CONFIGS["tiny_mh"], 64),
    "no_mlp": (tl.CONFIGS["tiny_nomlp"], 64),
    "D128": (dict(tl.CONFIGS["small"], D=128), 1600),
    "F44": (dict(tl.CONFIGS["small"], F=44), 1600),
}
BATCHES = (1, 3, 64, 65, 512)
MODES = (_cabi.MODE_FP32, _cabi.MODE_BF16, _cabi.MODE_F16, 7)  # 7: no such mode
STEPS = 300
BEAMS = (1, 4, 8)
QUERIES = ["listener_packed", "listener_workspace", "speller_packed", "speller_workspace", "beam_packed"] + [f"beam_workspace_k{k}" for k in BEAMS]


def dims(c, T, B):
    cell = _cabi.CELLS[c.get("unit", "LSTM")]
    ld = _cabi.ListenerDims(B, T, c["F"], c["H"], c["L"], cell)
    sd = _cabi.SpellerDims(B, T >> c["L"], 2 * c["H"], 2 * c["H"], c["sl"], c["V"], c["D"], c.get("heads", 1), int(not c.get("use_mlp", True)), cell)
    return ld, sd


def sizes(lib, ld, sd, mode):
    ld, sd = ctypes.byref(ld), ctypes.byref(sd)
    return [lib.las_listener_packed_bytes(ld, mode), lib.las_listener_workspace_bytes(ld, mode), lib.las_speller_packed_bytes(sd, mode),
            lib.las_speller_workspace_bytes(sd, STEPS, mode), lib.las_speller_beam_packed_bytes(sd, mode)] + \
           [lib.las_speller_beam_workspace_bytes(sd, STEPS, k, mode) for k in BEAMS]


def table(lib):
    out = {}
    for name, (c, T) in CONFIGS.items():
        for B in BATCHES:
            ld, sd = dims(c, T, B)
            for mode in MODES:
                out[f"{name} B={B} mode={mode}"] = sizes(lib, ld, sd, mode)
    return out


def load_table():
    with open(TABLE) as f:
        t = json.load(f)
    assert t["queries"] == QUERIES
    return t["sizes"]


def test_size_queries_match_the_pinned_table():
    expected = load_table()
    got = table(_cabi.load_library())
    assert sorted(got) == sorted(expected)
    wrong = {k: (got[k], expected[k]) for k in expected if got[k] != expected[k]}
    assert not wrong, wrong


def test_persistent_paths_are_in_the_table():
    """The table covers each layout: the tensor-core modes' sizes differ from the fp32 ones, and the persistent decoder's
    block differs from the generic one (the beam pack always holds the generic one)."""
    t = {k: dict(zip(QUERIES, v)) for k, v in load_table().items()}
    paper, shipped = t[f"paper B=64 mode={_cabi.MODE_BF16}"], t[f"shipped B=64 mode={_cabi.MODE_BF16}"]
    assert paper["speller_packed"] != paper["beam_packed"]
    assert shipped["speller_packed"] == shipped["beam_packed"]
    assert paper["listener_packed"] != t[f"paper B=64 mode={_cabi.MODE_FP32}"]["listener_packed"]


BAD_LISTENER = [None, dict(T=62), dict(L=0), dict(L=17), dict(H=0), dict(B=0), dict(cell=3)]
BAD_SPELLER = [None, dict(Hs=48), dict(sl=0), dict(sl=9), dict(heads=17), dict(heads=-1), dict(heads=2, no_mlp=1), dict(V=0), dict(D=0),
               dict(cell=3), dict(B=0)]


def _with(struct, kw):
    if kw is None:
        return None  # NULL dims
    s = type(struct).from_buffer_copy(struct)
    for k, v in kw.items():
        setattr(s, k, v)
    return ctypes.byref(s)


@pytest.mark.parametrize("mode", MODES)
def test_size_queries_return_zero_for_invalid_arguments(mode):
    lib = _cabi.load_library()
    ld, sd = dims(tl.CONFIGS["paper"], 1600, 64)
    for kw in BAD_LISTENER:
        assert lib.las_listener_packed_bytes(_with(ld, kw), mode) == 0, kw
        assert lib.las_listener_workspace_bytes(_with(ld, kw), mode) == 0, kw
    for kw in BAD_SPELLER:
        p = _with(sd, kw)
        assert lib.las_speller_packed_bytes(p, mode) == 0, kw
        assert lib.las_speller_workspace_bytes(p, STEPS, mode) == 0, kw
        assert lib.las_speller_beam_packed_bytes(p, mode) == 0, kw
        assert lib.las_speller_beam_workspace_bytes(p, STEPS, 4, mode) == 0, kw
    p = ctypes.byref(sd)
    assert lib.las_speller_workspace_bytes(p, -1, mode) == 0
    for steps, beam in ((0, 4), (-1, 4), (STEPS, 0), (STEPS, 33)):
        assert lib.las_speller_beam_workspace_bytes(p, steps, beam, mode) == 0, (steps, beam)


# ---- las_decode_io checks: las_pipeline_step's concurrent branch rejects what las_speller_decode rejects ------------------------

FAKE = 0x10000  # never dereferenced: every call below fails its argument checks first


def _decode_io(**kw):
    io = _cabi.DecodeIO()
    io.enc, io.logp = FAKE, FAKE
    for k, v in kw.items():
        setattr(io, k, v)
    return io


BAD_IO = [
    (dict(enc=None), 8, 1, "io->enc and io->logp are required"),
    (dict(logp=None), 8, 1, "io->enc and io->logp are required"),
    (dict(), 8, 3, "decode_mode 3 is not supported"),
    (dict(gt_dense=FAKE, gt_steps=7), 8, 1, "ground truth has 7 steps, 8 requested"),
    (dict(gt_index=FAKE, gt_steps=7), 8, 1, "ground truth has 7 steps, 8 requested"),
    (dict(h_state=FAKE), 8, 1, "h_state and c_state must be given together"),
    (dict(c_state=FAKE), 8, 1, "h_state and c_state must be given together"),
    (dict(word=FAKE), 8, 1, "word and context must be given together"),
    (dict(context=FAKE), 8, 1, "word and context must be given together"),
    (dict(early_exit=1), 8, 1, "<eos> early exit needs io->tokens"),
]


@pytest.mark.parametrize("io_kw,steps,decode_mode,msg", BAD_IO)
def test_pipeline_step_rejects_what_speller_decode_rejects(io_kw, steps, decode_mode, msg):
    lib = _cabi.load_library()
    mode = _cabi.MODE_BF16
    ld, sd = dims(tl.CONFIGS["paper"], 1600, 64)
    # the paper model at batch 64 runs the decoder and the next batch's listener concurrently
    assert lib.las_pipeline_overlaps(ctypes.byref(ld), ctypes.byref(sd), STEPS, mode) == 1
    io = _decode_io(**io_kw)
    big = 1 << 40
    st = lib.las_speller_decode(ctypes.byref(io), FAKE, ctypes.byref(sd), steps, decode_mode, mode, 1, FAKE, big, None)
    assert st == -1, st  # LAS_EINVAL
    decode_msg = lib.las_last_error()
    assert msg.encode() in decode_msg
    a = _cabi.PipelineArgs()
    a.dec_io = ctypes.pointer(io)
    a.speller_packed, a.speller_dims, a.steps, a.decode_mode, a.relu = FAKE, ctypes.pointer(sd), steps, decode_mode, 1
    a.speller_ws, a.speller_ws_bytes = FAKE, big
    a.x, a.listener_packed, a.listener_dims, a.enc, a.listener_ws, a.listener_ws_bytes = FAKE, FAKE, ctypes.pointer(ld), FAKE, FAKE, big
    assert lib.las_pipeline_step(ctypes.byref(a), mode, None) == -1
    assert lib.las_last_error() == decode_msg


if __name__ == "__main__":
    t = table(_cabi.load_library())
    rows = ",\n".join(f"  {json.dumps(k)}: {json.dumps(t[k])}" for k in sorted(t))
    sys.stdout.write(f'{{"queries": {json.dumps(QUERIES)},\n "sizes": {{\n{rows}\n}}}}\n')
