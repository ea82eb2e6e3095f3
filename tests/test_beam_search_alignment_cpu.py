"""Beam search's per-hypothesis attention and early exit without a GPU: the argument checks of the C ABI (las_beam_io.attn / attn_work /
early_exit / segment_steps / steps_done) and of the Python API."""
import ctypes

import pytest
import torch

import las_testlib as tl
from las_pytorch_b200 import _cabi
from test_beam_search_cpu import _dims, _io


def _call(io, steps=8):
    lib = _cabi.load_library()
    d = _dims()
    return lib.las_speller_beam_search(ctypes.byref(io), ctypes.c_void_p(0x5000), ctypes.byref(d), steps, 0, 1, ctypes.c_void_p(0x6000),
                                       1 << 20, None)


@pytest.mark.parametrize("kw,msg", [
    (dict(attn=0x7000), b"attn_work"),
    (dict(early_exit=1), b"steps_done"),
    (dict(segment_steps=-1), b"segment_steps"),
    (dict(early_exit=1, steps_done=0x8000, segment_steps=-3), b"segment_steps"),
])
def test_new_fields_are_checked_before_touching_the_device(kw, msg):
    assert _call(_io(**kw)) == -1  # LAS_EINVAL
    assert msg in _cabi.load_library().las_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the path that ends at the missing device")
def test_valid_new_fields_get_past_the_checks():
    for kw in (dict(attn=0x7000, attn_work=0x9000), dict(early_exit=1, steps_done=0x8000), dict(early_exit=1, steps_done=0x8000, segment_steps=5),
               dict(attn_work=0x9000)):
        assert _call(_io(**kw)) != -1, kw


def test_abi_version_is_7():
    assert _cabi.ABI_VERSION == 7 and _cabi.load_library().las_abi_version() == 7
    assert [f for f, _ in _cabi.BeamIO._fields_][-5:] == ["attn", "attn_work", "early_exit", "segment_steps", "steps_done"]


@pytest.mark.parametrize("kw", [dict(return_attention=1), dict(return_attention=None), dict(early_exit=1), dict(early_exit="yes"),
                                dict(early_exit=0.0)])
def test_python_flags_must_be_bools(kw):
    las = tl.build_model("tiny", max_label_len=6)
    with pytest.raises(ValueError):
        las.speller.beam_search(torch.zeros(2, 4, 32), **kw)  # on the CPU: the check comes before the device is needed
    with pytest.raises(ValueError):
        las.beam_search(torch.zeros(2, 16, 40), **kw)


def test_python_valid_flags_reach_the_missing_device():
    las = tl.build_model("tiny", max_label_len=6)
    las.speller.early_exit = True  # greedy decoding's switch: beam search does not read it
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        las.speller.beam_search(torch.zeros(2, 4, 32), return_attention=True, early_exit=True)
    assert not hasattr(las.speller, "last_steps_done")
