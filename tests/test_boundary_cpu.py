"""Host-side boundary checks that need no GPU: ABI surface, state_dict layout, error behaviour."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import las_testlib as tl
import las_pytorch_b200 as lp
from las_pytorch_b200 import _cabi


def header_functions():
    src = open(os.path.join(tl.ROOT, "include", "las_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(las_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _cabi.load_library()
    names = header_functions()
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/las_b200.h but not exported by liblas_b200.so"
    assert sorted(_cabi.PROTOTYPES) == names, "ctypes prototypes and header declarations differ"
    assert lib.las_abi_version() == _cabi.ABI_VERSION


def test_size_queries_run_on_host():
    lib = _cabi.load_library()
    d = _cabi.ListenerDims(64, 1600, 40, 256, 3)
    for mode in (_cabi.MODE_FP32,):
        assert lib.las_listener_packed_bytes(ctypes.byref(d), mode) >= 4 * (2048 * 80 + 2 * 2048 * 1024 + 3 * 2048 * 256)
        assert lib.las_listener_workspace_bytes(ctypes.byref(d), mode) >= 4 * 64 * 800 * 2048
    bad = _cabi.ListenerDims(2, 62, 40, 16, 2)  # 62 is not divisible by 4
    assert lib.las_listener_packed_bytes(ctypes.byref(bad), 0) == 0
    assert b"not divisible" in lib.las_last_error()
    s = _cabi.SpellerDims(64, 200, 512, 512, 2, 30, 64)
    assert lib.las_speller_packed_bytes(ctypes.byref(s), 0) >= 4 * 4_260_000
    bad_s = _cabi.SpellerDims(4, 10, 64, 48, 2, 30, 16)  # Hs != E
    assert lib.las_speller_packed_bytes(ctypes.byref(bad_s), 0) == 0
    assert b"must equal" in lib.las_last_error()


def test_debug_options_take_documented_values_and_reject_the_rest():
    """las_debug_set_option accepts each key listed in include/las_b200.h with the values listed there, and returns LAS_EINVAL
    with a message naming the key for any other key or value: a tool that names a retired or mistyped option fails instead of
    timing the default kernel twice."""
    lib = _cabi.load_library()
    overlap = 0 if os.environ.get("LAS_B200_NO_OVERLAP", "") not in ("", "0") else 1  # as _cabi.load_library leaves key 6
    defaults = {2: 1, 6: overlap, 8: 0, 9: 0, 11: 1, 12: 1, 13: 0, 19: 1, **{20 + l: 0 for l in range(8)}}
    values = {2: [0, 1], 6: [0, 1], 8: [0, 1], 9: [0, 16, 32, 64], 11: [0, 1], 12: [0, 1], 13: [0, 1, 2, 4, 8], 19: [0, 1],
              **{20 + l: [0, 1, 160] for l in range(8)}}
    try:
        for key, vals in values.items():
            for v in vals:
                assert lib.las_debug_set_option(key, v) == 0, (key, v)
    finally:
        for key, v in defaults.items():
            assert lib.las_debug_set_option(key, v) == 0, (key, v)
    rejected = [(k, 1) for k in (1, 4, 7, 10, 15, 16, 18)] + [(k, 0) for k in (0, 3, 14, 17, 28, 99, -1)]
    rejected += [(5, 0), (5, 1), (5, 4), (5, 16384), (2, 2), (11, 2), (11, 3), (19, 2), (13, 3), (13, 16), (9, 8), (6, 2), (8, -1), (12, 2), (20, -1)]
    for key, v in rejected:
        assert lib.las_debug_set_option(key, v) == -1, (key, v)  # LAS_EINVAL
        assert f"key {key} ".encode() in lib.las_last_error(), (key, v)


@pytest.mark.parametrize("cfg,count", [("small", 2_004_126), ("paper", 10_303_646)])
def test_state_dict_layout_matches_reference(cfg, count):
    """SURVEY.md A.2: key names, order within an LSTM, shapes and parameter counts."""
    c = tl.CONFIGS[cfg]
    las = tl.build_model(cfg, max_label_len=10)
    sd = las.state_dict()
    assert sum(v.numel() for v in sd.values()) == count
    H, V, D = c["H"], c["V"], c["D"]
    keys = list(sd)
    assert keys[:8] == [f"listener.pLSTM_layer0.BLSTM.{n}" for n in (
        "weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0",
        "weight_ih_l0_reverse", "weight_hh_l0_reverse", "bias_ih_l0_reverse", "bias_hh_l0_reverse")]
    assert sd["listener.pLSTM_layer0.BLSTM.weight_ih_l0"].shape == (4 * H, 80)
    assert sd["listener.pLSTM_layer1.BLSTM.weight_ih_l0_reverse"].shape == (4 * H, 4 * H)
    assert sd["speller.rnn_layer.weight_ih_l0"].shape == (8 * H, V + 2 * H)
    assert sd["speller.rnn_layer.weight_ih_l1"].shape == (8 * H, 2 * H)
    assert sd["speller.attention.phi.weight"].shape == (D, 2 * H)
    assert sd["speller.attention.psi.bias"].shape == (D,)
    assert sd["speller.character_distribution.weight"].shape == (V, 4 * H)
    assert all(v.dtype == torch.float32 for v in sd.values())


def test_loads_reference_state_dict_strictly():
    g = np.load(os.path.join(tl.GOLDEN_DIR, "tiny_tf_g3.npz"))
    sd = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("w:")}
    las = tl.build_model("tiny", max_label_len=6, seed=1)
    las.load_state_dict(sd, strict=True)
    assert torch.equal(las.speller.rnn_layer.weight_hh_l1, sd["speller.rnn_layer.weight_hh_l1"])
    pkg = las.serialize(None, epoch=3, tr_loss=1.0, val_loss=2.0)
    assert set(pkg) == {"einput", "ehidden", "elayer", "edropout", "etype", "dvocab_size", "dhidden", "dlayer",
                        "state_dict", "optim_dict", "epoch", "tr_loss", "val_loss"}
    assert pkg["etype"] is torch.nn.LSTM and pkg["dvocab_size"] == 30


def test_constructor_contract():
    # kwargs splatted from the YAML are swallowed (model/las_model.py:105,153)
    lis = lp.Listener(input_feature_dim=40, hidden_size=16, num_layers=2, rnn_unit="LSTM", use_gpu=True, dropout=0.0, bidirectional=True)
    assert (lis.input_feature_dim, lis.hidden_size, lis.num_layers, lis.rnn_unit, lis.dropout_rate) == (40, 16, 2, "LSTM", 0.0)
    sp = lp.Speller(30, 32, "LSTM", 2, 7, True, 16, "relu", 16, 1, 1, use_gpu=False, bidirectional=True)
    assert (sp.label_dim, sp.hidden_size, sp.num_layers, sp.max_label_len, sp.decode_mode) == (30, 32, 2, 7, 1)
    assert sp.float_type is torch.FloatTensor
    with pytest.raises(AssertionError):
        lp.Listener(40, 16, 0, "LSTM", True)
    with pytest.raises(ValueError):
        lp.Speller(30, 48, "LSTM", 2, 7, True, 16, "relu", 16, 1, 1)  # Hs != 2H
    gru = lp.Listener(40, 16, 2, "GRU", True)  # rnn_unit as the reference resolves it: getattr(nn, rnn_unit.upper())
    assert gru.pLSTM_layer0.BLSTM.weight_ih_l0.shape == (3 * 16, 80) and gru.pLSTM_layer1.BLSTM.weight_hh_l0_reverse.shape == (48, 16)
    assert list(gru.state_dict()) == list(torch.nn.GRU(80, 16, 1, bidirectional=True).state_dict().__class__(
        (f"pLSTM_layer{i}.BLSTM.{k}", None) for i in range(2) for k in torch.nn.GRU(80, 16, 1, bidirectional=True).state_dict()))
    assert lp.Listener(40, 16, 2, "GRU", True, precision="bf16").cell == "GRU"  # both modes take GRU / RNN cells
    with pytest.raises(NotImplementedError):
        lp.Listener(40, 16, 2, "QRNN", True)


def test_no_cpu_fallback_and_single_rng_draw():
    las = tl.build_model("tiny", max_label_len=4)
    x = torch.randn(2, 16, 40)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        las.listener(x)
    enc = torch.randn(2, 4, 32)
    np.random.seed(5)
    expect = np.random.RandomState(5)
    expect.random_sample()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        las.speller(enc, ground_truth=None, teacher_force_rate=0.9)
    # exactly one draw from numpy's global RNG per Speller.forward call (model/las_model.py:189)
    assert np.random.random_sample() == expect.random_sample()


def test_missing_library_fails_loudly(tmp_path):
    with pytest.raises(_cabi.LasB200Error, match="no CPU fallback"):
        _cabi.load_library(str(tmp_path / "nope.so"))


def test_product_does_not_import_oracle():
    for root, _, files in os.walk(os.path.join(tl.ROOT, "las_pytorch_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                assert "oracle" not in open(os.path.join(root, f)).read(), f"{f} references oracle/"


def test_checkpoint_package_roundtrip(tmp_path):
    """SURVEY.md 8 row f3: reference-format package (train.py:83-90,181-201), incl. a DataParallel `module.` prefix."""
    from las_pytorch_b200 import checkpoint

    las = tl.build_model("tiny", max_label_len=9, seed=5)
    path = str(tmp_path / "las-epoch3.pth.tar")
    checkpoint.save_package(las, path, optimizer=None, epoch=3, tr_loss=1.5, val_loss=2.5)
    las2, pkg = checkpoint.load_package(path, mlp_dim_in_attention=16, max_label_len=9)
    assert pkg["epoch"] == 3 and pkg["ehidden"] == 16 and pkg["dhidden"] == 32
    for (k1, v1), (k2, v2) in zip(las.state_dict().items(), las2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    pkg["state_dict"] = {"module." + k: v for k, v in pkg["state_dict"].items()}
    las3, _ = checkpoint.load_package(pkg, las=tl.build_model("tiny", max_label_len=9, seed=1))
    assert torch.equal(las3.listener.pLSTM_layer1.BLSTM.weight_hh_l0_reverse, las.listener.pLSTM_layer1.BLSTM.weight_hh_l0_reverse)


def test_models_build_from_the_shipped_yaml_sections():
    """train.py:73-74 builds the models with Listener(**params["model"]["listener"]) / Speller(**params["model"]["speller"]); the
    shipped config (config/librispeech-config.yaml:13-34) carries keys the classes swallow (dropout, bidirectional)."""
    import las_pytorch_b200 as lp

    listener_cfg = dict(input_feature_dim=40, hidden_size=512, num_layers=3, dropout=0.0, bidirectional=True, rnn_unit="LSTM", use_gpu=True)
    speller_cfg = dict(hidden_size=1024, num_layers=2, bidirectional=True, rnn_unit="LSTM", vocab_size=30, multi_head=1, decode_mode=1,
                       use_mlp_in_attention=True, mlp_dim_in_attention=64, mlp_activate_in_attention="relu", listener_hidden_size=512,
                       max_label_len=576)
    las = lp.LAS(lp.Listener(**listener_cfg), lp.Speller(**speller_cfg))
    sd = las.state_dict()
    assert sd["listener.pLSTM_layer2.BLSTM.weight_ih_l0_reverse"].shape == (2048, 2048)
    assert sd["speller.rnn_layer.weight_ih_l0"].shape == (4096, 30 + 1024)
    assert sd["speller.character_distribution.weight"].shape == (30, 2048)
    assert sum(v.numel() for v in sd.values()) == sum(p.numel() for p in las.parameters())


def test_reference_written_package_loads():
    """Row f3 against the real thing: tests/golden/ref_package_tiny*.pth.tar were written by the REFERENCE's LAS.serialize +
    torch.save (model/las_model.py:42-63, train.py:181-192; tests/golden/make_golden.py extras).  `etype` is the pickled class
    nn.LSTM (the :49/:54 duplicate-key quirk); the second file carries nn.DataParallel's `module.` key prefix."""
    from las_pytorch_b200 import checkpoint

    las, pkg = checkpoint.load_package(os.path.join(tl.GOLDEN_DIR, "ref_package_tiny.pth.tar"), max_label_len=8)
    assert pkg["etype"] is torch.nn.LSTM and pkg["epoch"] == 7 and pkg["tr_loss"] == 1.25 and pkg["val_loss"] == 1.5
    assert pkg["optim_dict"]["param_groups"][0]["lr"] == 1e-3
    c = tl.CONFIGS["tiny"]
    assert (las.listener.hidden_size, las.listener.num_layers, las.speller.hidden_size, las.speller.num_layers, las.speller.label_dim) == \
        (c["H"], c["L"], 2 * c["H"], c["sl"], c["V"])
    assert las.speller.attention.preprocess_mlp_dim == c["D"] and las.speller.attention.multi_head == 1
    for k, v in pkg["state_dict"].items():
        assert torch.equal(las.state_dict()[k], v)
    # our serialize() writes the same key set, with the same `etype` value, as the reference's
    ours = las.serialize(None, 7, 1.25, 1.5)
    assert sorted(ours) == sorted(pkg) and ours["etype"] is pkg["etype"]
    assert list(ours["state_dict"]) == list(pkg["state_dict"])
    las_dp, _ = checkpoint.load_package(os.path.join(tl.GOLDEN_DIR, "ref_package_tiny_dataparallel.pth.tar"), max_label_len=8)
    for a, b in zip(las.state_dict().values(), las_dp.state_dict().values()):
        assert torch.equal(a, b)
    # the variants' hyper-parameters the package does not record are read off the state_dict
    mh = tl.build_model("tiny_mh", max_label_len=4, seed=3)
    las_mh, _ = checkpoint.load_package(mh.serialize(None, 0, None, None), max_label_len=4)
    assert las_mh.speller.attention.multi_head == 2 and las_mh.speller.attention.preprocess_mlp_dim == 16
    gru = tl.build_model("tiny_gru", max_label_len=4, seed=3)
    las_gru, _ = checkpoint.load_package(gru.serialize(None, 0, None, None), max_label_len=4)
    assert las_gru.speller.cell == "GRU" and las_gru.listener.cell == "GRU"


def test_oracle_solver_losses_match_the_reference_values():
    """Row f1: the oracle's restatement of label_smoothing_loss / NLLLoss(ignore_index=0) / LetterErrorRate
    (solver/solver.py:11-24,33-45,62) against values the reference's own functions produced (ref_solver_losses.npz)."""
    from las_pytorch_b200 import solver as our_solver
    from oracle import las_oracle as O

    g = np.load(os.path.join(tl.GOLDEN_DIR, "ref_solver_losses.npz"))
    logp, lab, lens = g["logp"], g["labels"], g["lens"]
    V = logp.shape[-1]
    zero_pad = np.eye(V)[lab]
    lab0 = lab.copy()
    for b, n in enumerate(lens):
        zero_pad[b, n:] = 0
        lab0[b, n:] = 0
    pad0 = np.eye(V)[lab0]
    for ls in (0.1, 0.3):
        assert abs(O.label_smoothing_loss(logp, zero_pad, ls) - float(g[f"ls_zero_pad_{ls}"])) < 1e-5
        assert abs(O.label_smoothing_loss(logp, pad0, ls) - float(g[f"ls_pad0_{ls}"])) < 1e-5
    assert abs(O.nll_loss_ignore0(logp, lab0) - float(g["nll_ignore0"])) < 1e-5
    assert np.allclose(our_solver.LetterErrorRate(logp.argmax(-1), lab0), g["ler"])


def test_packed_weight_cache_keys_follow_the_tensors_handed_to_the_pack_call():
    """ADVICE r1 (high): under nn.DataParallel replicas share the original's cache object and `.parameters()` is empty on a
    replica, so the key must come from the tensors themselves, entries must be per device, and replicas must never reuse one."""
    from las_pytorch_b200.las_model import _Cache, _weight_tensors

    las = tl.build_model("tiny", max_label_len=4, seed=3)
    ts = _weight_tensors(las.speller)
    assert len(ts) == len(list(las.speller.parameters())) > 0
    assert las.speller._replicate_for_data_parallel()._cache is las.speller._cache  # shallow __dict__ copy: ONE cache object
    replica = las.speller.rnn_layer._replicate_for_data_parallel()
    assert list(replica.parameters()) == [] and getattr(replica, "_is_replica", False)
    for name, p in las.speller.rnn_layer._parameters.items():  # what nn.parallel.replicate does: plain tensors in _parameters
        replica._parameters[name] = p.detach().clone()
    assert len(_weight_tensors(replica)) == len(las.speller.rnn_layer._parameters)
    k1 = _Cache.tensors_key(ts, 0)
    with torch.no_grad():
        ts[0].add_(1.0)
    assert _Cache.tensors_key(ts, 0) != k1  # an in-place update (optimizer step, load_state_dict) changes the key
    cache = _Cache()
    dev = torch.device("cuda", 0)
    cache.store(dev, 0, k1, "image")
    assert cache.lookup(dev, 0, k1, is_replica=False) == "image"
    assert cache.lookup(dev, 0, k1, is_replica=True) is None           # replicas always repack
    assert cache.lookup(torch.device("cuda", 1), 0, k1, False) is None  # entries are per device
    cache.store(torch.device("cuda", 1), 0, k1, "image1")
    assert cache.lookup(dev, 0, k1, False) == "image"                   # ... and a device replaces only its own
    cache.invalidate()
    assert cache.lookup(dev, 0, k1, False) is None
    # modules stay deep-copyable and picklable (EMA copies, torch.save(model)): a copied cache starts empty
    import copy
    import pickle

    cache.store(dev, 0, k1, "image")
    las2 = copy.deepcopy(las)
    assert las2.speller._cache is not las.speller._cache and las2.speller._cache.packed == {}
    assert pickle.loads(pickle.dumps(cache)).packed == {}
