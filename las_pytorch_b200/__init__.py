"""las_pytorch_b200 -- B200-native (sm_100a) LAS forward hot path behind jiwidi/las-pytorch's model API.

    from las_pytorch_b200 import Listener, Speller, LAS        # same signatures as model/las_model.py

The arithmetic lives in `liblas_b200.so` (hand-written CUDA, C ABI in include/las_b200.h); build it with
`python -m las_pytorch_b200.build`.  There is no CPU fallback.
"""
from .las_model import LAS, Attention, BeamSearchResult, Listener, Speller, pBLSTMLayer  # noqa: F401
from .functions import CreateOnehotVariable, TimeDistributed  # noqa: F401
from ._cabi import LasB200Error, load_library  # noqa: F401

__all__ = [
    "LAS", "Attention", "BeamSearchResult", "Listener", "Speller", "pBLSTMLayer",
    "CreateOnehotVariable", "TimeDistributed", "LasB200Error", "load_library",
]
