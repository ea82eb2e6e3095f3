"""Host-side mirror of the reference's `model/las_model.py` for the forward hot path.

Same class names, constructor arguments, `forward` signatures, return structures and `state_dict` layout as
/root/reference/model/las_model.py (LAS :24-63, pBLSTMLayer :66-91, Listener :96-134, Speller :138-238,
Attention :249-318); the arithmetic is done by the sm_100a kernels behind the C ABI (include/las_b200.h).
torch is used only for device memory, the current stream and parameter storage.

Extra keyword accepted everywhere the reference swallows **kwargs: `precision` = "fp32" | "bf16" | "fp16"
(LAS_MODE_FP32 / LAS_MODE_BF16 / LAS_MODE_F16 -- the tensor-core kernels with bf16 or IEEE fp16 GEMM operands; default from
$LAS_B200_PRECISION, else "fp32").

Variants of the reference classes -- multi_head > 1 (with attention.dim_reduce), use_mlp_in_attention=False, GRU / RNN cells
(`rnn_unit`; the reference does getattr(nn, rnn_unit.upper()), :69,156) and cells too wide for the persistent decoder (the shipped
config's 1024) -- run in both modes; in the bf16 mode their GEMMs (input projections, [x | h] . [W_ih | W_hh]^T per cell and step,
psi) are tcgen05 GEMMs over bf16 operands and everything else stays fp32 (the generic tensor-core path, csrc/las_api.cu).  decode_mode 2 samples the fed-back word on the device from the reference's distribution
(Categorical(probs=log-probs), SURVEY.md A.5.6) with a counter-based generator seeded from torch's global generator, so runs are
reproducible under torch.manual_seed but not draw-for-draw equal to the reference.  Not on this path: training/backward.
"""
from __future__ import annotations

import collections
import ctypes as C
import math
import os
import threading

import numpy as np
import torch
import torch.nn as nn

from . import _cabi
from ._cabi import BeamIO, DecodeIO, ListenerDims, LstmWeights, SpellerDims, SpellerWeights, check, current_stream_ptr, ptr
from .params import LinearWeights, LSTMWeights

_MODES = {"fp32": _cabi.MODE_FP32, "bf16": _cabi.MODE_BF16, "fp16": _cabi.MODE_F16}


def _default_precision():
    return os.environ.get("LAS_B200_PRECISION", "fp32")


def _mode_of(precision):
    if precision not in _MODES:
        raise ValueError(f"precision must be one of {sorted(_MODES)}, got {precision!r}")
    return _MODES[precision]


def _require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(
            f"{what} is on {t.device}: las_pytorch_b200 runs on a B200 (sm_100a) only and has no CPU fallback"
        )


def _f32c(t):
    return t.detach().to(torch.float32).contiguous()


def _weight_tensors(*holders):
    """The tensors a pack call will read, in registration order.  `_parameters` (not `.parameters()`) on purpose: an
    nn.DataParallel replica (train.py:76-78) keeps its per-device broadcast copies there as plain tensors, and
    `.parameters()` yields nothing on a replica."""
    out = []
    for h in holders:
        for m in h.modules():
            out.extend(t for t in m._parameters.values() if t is not None)
    return out


class _Cache:
    """Packed-weight / workspace cache.  One packed image per (device, mode), valid while the tensors that were packed are still
    the module's tensors: the key is (data_ptr, version counter, device) of every weight actually handed to the pack call.

    nn.DataParallel shallow-copies a module's __dict__ into every replica, so replicas on all devices share THIS object with
    the original: entries are per device, a device only ever replaces its own entry, and mutation is locked.  A replica's
    weights are fresh broadcast copies each forward (same addresses can come back from the caching allocator with new contents,
    version 0), so replicas never reuse a packed image: they repack on every call (a few pack kernels, ~30 MB at paper size).
    In-place writes through `.data` (nn.init.*_(p.data), p.data.copy_()) do not bump the version counter: call
    `invalidate()` (LAS.invalidate_packed_weights) after such an update."""

    def __init__(self):
        self.packed = {}
        self.work = {}
        self.lock = threading.Lock()
        self.enqueue_locks = {}

    # copy.deepcopy(model) / pickling a module (torch.save(model)) must not drag device buffers or locks along: a copy starts empty
    def __deepcopy__(self, memo):
        return _Cache()

    def __reduce__(self):
        return (_Cache, ())

    def enqueue_lock(self, device):
        """Held while one forward's kernels are being enqueued: the workspace of a (module, device, stream) is reused by every call,
        which is only safe if two host threads never interleave their launches on it (the work itself is asynchronous; the lock
        covers host-side enqueue time only).  One lock per device, so DataParallel's per-GPU threads do not serialise each other."""
        with self.lock:
            return self.enqueue_locks.setdefault(device.index, threading.RLock())

    @staticmethod
    def tensors_key(tensors, mode):
        return (mode,) + tuple((t.data_ptr(), t._version, t.device.index) for t in tensors)

    def lookup(self, device, mode, key, is_replica):
        if is_replica:
            return None
        with self.lock:
            hit = self.packed.get((device.index, mode))
        return hit[1] if hit is not None and hit[0] == key else None

    def store(self, device, mode, key, packed):
        with self.lock:
            self.packed[(device.index, mode)] = (key, packed)

    def invalidate(self):
        with self.lock:
            self.packed.clear()

    def workspace(self, key, nbytes, device):
        with self.lock:
            buf = self.work.get(key)
            if buf is None or buf.numel() < nbytes:
                buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
                self.work[key] = buf
        return buf


def _lstm_weight_array(holder, layers, directions):
    """Host array of las_lstm_weights (device pointers) + the tensors kept alive."""
    arr = (LstmWeights * (layers * directions))()
    keep = []
    for l in range(layers):
        for d in range(directions):
            sfx = "_reverse" if d == 1 else ""
            ts = [_f32c(getattr(holder, f"{n}_l{l}{sfx}")) for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            keep.extend(ts)
            e = arr[l * directions + d]
            e.w_ih, e.w_hh, e.b_ih, e.b_hh = (t.data_ptr() for t in ts)
    return arr, keep


class _Call:
    """Marshalled arguments of one C-ABI call: ctypes structs, the tensors they point into (kept alive here) and the outputs."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


def _prepare_listener(x, holders, input_feature_dim, hidden_size, mode, cache, lengths=None, cell="LSTM", is_replica=False):
    """Checks, packed weights, workspace and output buffers of one listener call (the caller holds cache.enqueue_lock)."""
    _require_cuda(x, "input_x")
    lib = _cabi.load_library()
    x = _f32c(x)
    b, t, f = x.shape
    if f != input_feature_dim:
        raise RuntimeError(f"input feature dim {f} != {input_feature_dim}")
    nl = len(holders)
    dims = ListenerDims(b, t, f, hidden_size, nl, _cabi.CELLS[cell])
    if t % (1 << nl) != 0:
        # the reference fails inside `view` (model/las_model.py:87) with a RuntimeError; so do we
        raise RuntimeError(
            f"shape '[{b}, {t >> 1}, {f * 2}]' is invalid: timestep {t} is not divisible by 2^{nl} "
            "(model/las_model.py:86-87 halves the time axis in every layer)"
        )
    if lengths is not None and lengths.numel() != b:
        raise RuntimeError(f"input_lengths has {lengths.numel()} entries for a batch of {b}")
    st = current_stream_ptr(x.device)
    tensors = _weight_tensors(*holders)
    for w in tensors:
        _require_cuda(w, "listener weight")
        if w.device != x.device:
            raise RuntimeError(f"listener weights are on {w.device}, input_x on {x.device}")
    key = _Cache.tensors_key(tensors, mode)
    packed = cache.lookup(x.device, mode, key, is_replica)
    if packed is None:
        arr = (LstmWeights * (2 * nl))()
        keep = []
        for l, h in enumerate(holders):
            a1, k1 = _lstm_weight_array(h, 1, 2)
            keep.extend(k1)
            for d in range(2):
                arr[2 * l + d] = a1[d]
        nbytes = lib.las_listener_packed_bytes(C.byref(dims), mode)
        packed = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=x.device)
        check(lib.las_listener_pack(arr, C.byref(dims), mode, ptr(packed), packed.numel(), st))
        cache.store(x.device, mode, key, packed)
        del keep
    ws_bytes = lib.las_listener_workspace_bytes(C.byref(dims), mode)
    ws = cache.workspace(("listener", x.device, mode, st.value), ws_bytes, x.device)
    enc = torch.empty(b, t >> nl, 2 * hidden_size, dtype=torch.float32, device=x.device)
    lens = enc_lens = None
    if lengths is not None:
        lens = lengths.to(device=x.device, dtype=torch.int32).contiguous()
        enc_lens = torch.empty(b, dtype=torch.int32, device=x.device)
    return _Call(lib=lib, x=x, dims=dims, packed=packed, ws=ws, enc=enc, lens=lens, enc_lens=enc_lens, mode=mode, st=st)


def _run_listener(x, holders, input_feature_dim, hidden_size, mode, cache, lengths=None, cell="LSTM", is_replica=False):
    """x [B,T,F] -> [B, T/2^L, 2H] through `len(holders)` pyramid layers.  With `lengths` ([B] valid frames; extension)
    returns (enc, enc_lengths [B] int32)."""
    _require_cuda(x, "input_x")
    with torch.cuda.device(x.device), cache.enqueue_lock(x.device):
        c = _prepare_listener(x, holders, input_feature_dim, hidden_size, mode, cache, lengths, cell, is_replica)
        if c.lens is None:
            check(c.lib.las_listener_forward(ptr(c.x), ptr(c.packed), C.byref(c.dims), mode, ptr(c.enc), ptr(c.ws), c.ws.numel(), c.st))
            return c.enc
        check(c.lib.las_listener_forward_masked(ptr(c.x), ptr(c.lens), ptr(c.packed), C.byref(c.dims), mode, ptr(c.enc), ptr(c.enc_lens),
                                                ptr(c.ws), c.ws.numel(), c.st))
    return c.enc, c.enc_lens


class LAS(nn.Module):
    """model/las_model.py:24-63."""

    def __init__(self, listener, speller):
        super().__init__()
        self.listener = listener
        self.speller = speller

    def forward(self, batch_data, batch_label, teacher_force_rate, is_training=True, input_lengths=None, nll_labels=None):
        """`input_lengths` ([B] valid frames per utterance) is an extension: the reference's collate_fn computes it
        (utils/data.py:146) and train.py:117 drops it.  When given, the BLSTMs and the attention skip the padding.
        `nll_labels` ([B,S'] label indices; extension) -> `self.speller.last_nll_terms` (see Speller.forward)."""
        enc_lengths = None
        if not is_training and nll_labels is None and self._chunk_pipelining_applies(batch_data):
            return self._forward_chunk_pipelined(batch_data, input_lengths)
        if input_lengths is None:
            listener_feature = self.listener(batch_data)
        else:
            listener_feature, enc_lengths = self.listener(batch_data, input_lengths=input_lengths)
        if is_training:
            raw_pred_seq, attention_record = self.speller(
                listener_feature, ground_truth=batch_label, teacher_force_rate=teacher_force_rate, enc_lengths=enc_lengths,
                nll_labels=nll_labels
            )
        else:
            raw_pred_seq, attention_record = self.speller(listener_feature, ground_truth=None, teacher_force_rate=0,
                                                          enc_lengths=enc_lengths, nll_labels=nll_labels)
        return raw_pred_seq, attention_record

    def beam_search(self, batch_data, beam_width=8, nbest=1, length_penalty=0.0, input_lengths=None, return_attention=False,
                    early_exit=False):
        """Beam-search decoding (extension; the reference decodes greedily): the listener (with the length mask when
        `input_lengths` is given), then `Speller.beam_search` over `max_label_len` steps.  Returns a BeamSearchResult, or with
        `return_attention` a BeamSearchAlignedResult; `early_exit` as in Speller.beam_search."""
        _check_beam_args(beam_width, nbest, length_penalty, self.speller.max_label_len, return_attention, early_exit)
        enc_lengths = None
        if input_lengths is None:
            listener_feature = self.listener(batch_data)
        else:
            listener_feature, enc_lengths = self.listener(batch_data, input_lengths=input_lengths)
        return self.speller.beam_search(listener_feature, beam_width=beam_width, nbest=nbest, length_penalty=length_penalty,
                                        enc_lengths=enc_lengths, return_attention=return_attention, early_exit=early_exit)

    # ---- large free-running batches: the serving pipeline applied INSIDE one forward call ------------------------------------
    CHUNK = 64  # utterances per persistent decoder launch group (one attention CTA each next to the 64 LSTM CTAs)

    def _chunk_pipelining_applies(self, x):
        """A free-running batch of more than one decoder launch group (BASELINE config 5: 512 utterances on one GPU) is decoded
        64 utterances at a time anyway; when the concurrent schedule covers the model, chunk i+1's listener runs under chunk i's
        decoder.  An utterance's result does not depend on the batch it is in (bit-exact in both modes), so the outputs are the same."""
        sp, lis = self.speller, self.listener
        if not x.is_cuda or x.dim() != 3 or x.size(0) <= self.CHUNK or getattr(sp, "early_exit", False):
            return False
        if lis.precision == "fp32" or sp.precision != lis.precision or x.size(1) % (1 << lis.num_layers) != 0:
            return False
        lib = _cabi.load_library()
        ld = ListenerDims(self.CHUNK, x.size(1), x.size(2), lis.hidden_size, lis.num_layers, _cabi.CELLS[lis.cell])
        sd = sp._dims(self.CHUNK, x.size(1) >> lis.num_layers, 2 * lis.hidden_size)
        return bool(lib.las_pipeline_overlaps(C.byref(ld), C.byref(sd), int(sp.max_label_len), _mode_of(sp.precision)))

    def _forward_chunk_pipelined(self, x, input_lengths):
        np.random.random_sample()  # Speller.forward's one draw from numpy's global RNG per call (model/las_model.py:189)
        pipe = ServingPipeline(self, want_attention=True)
        outs = []
        for i in range(0, x.size(0), self.CHUNK):
            r = pipe.submit(x[i:i + self.CHUNK], None if input_lengths is None else input_lengths[i:i + self.CHUNK])
            if r is not None:
                outs.append(r)
        outs.append(pipe.flush())
        logp = torch.cat([o.logp for o in outs], dim=1)
        attn = torch.cat([o.attn for o in outs], dim=1)
        sp = self.speller
        sp.last_tokens = torch.cat([o.tokens for o in outs], dim=1)
        sp.last_logp = logp
        sp.last_nll_terms = sp.last_steps_done = None
        return list(logp.unbind(0)), [[a] for a in attn.unbind(0)]

    def serve(self, want_attention=True):
        """Cross-batch serving pipeline (extension; free-running decoding = the reference's is_training=False path,
        model/las_model.py:36-39).  `pipe.submit(x)` enqueues batch i+1's Listener UNDER batch i's decoder and returns batch i's
        results; `pipe.flush()` decodes the last batch.  Same numbers as calling `forward` batch by batch."""
        return ServingPipeline(self, want_attention)

    def invalidate_packed_weights(self):
        """Drops every cached kernel-layout weight image.  The caches follow parameter identity and version counters, which
        `load_state_dict`, optimizer steps and `.to()` change; an in-place write through `.data` does not -- call this after one."""
        for m in self.modules():
            c = getattr(m, "_cache", None)
            if isinstance(c, _Cache):
                c.invalidate()

    def serialize(self, optimizer, epoch, tr_loss, val_loss):
        """Checkpoint package with the reference's keys (model/las_model.py:42-63; "etype" is written twice
        there, the speller's value wins -- reproduced)."""
        package = {
            "einput": self.listener.input_feature_dim,
            "ehidden": self.listener.hidden_size,
            "elayer": self.listener.num_layers,
            "edropout": self.listener.dropout_rate,
            "dvocab_size": self.speller.label_dim,
            "dhidden": self.speller.hidden_size,
            "dlayer": self.speller.num_layers,
            "etype": self.speller.rnn_unit,
            "state_dict": self.state_dict(),
            "optim_dict": optimizer.state_dict() if optimizer is not None else None,
            "epoch": epoch,
        }
        if tr_loss is not None:
            package["tr_loss"] = tr_loss
            package["val_loss"] = val_loss
        return package


class ServingResult:
    """Outputs of one decoded batch (device tensors, valid once the stream they were enqueued on reaches them)."""

    def __init__(self, logp, attn, tokens, steps_done=None):
        self.logp, self.attn, self.tokens, self.steps_done = logp, attn, tokens, steps_done

    @property
    def raw_pred_seq(self):  # the reference's return structure (model/las_model.py:213,238)
        return list(self.logp.unbind(0))

    @property
    def attention_record(self):  # per step: one [B,U] tensor per head (model/las_model.py:214,292,299)
        if self.attn is None:
            return None
        return [[a] if a.dim() == 2 else list(a.unbind(0)) for a in self.attn.unbind(0)]


class ServingPipeline:
    """Two batches in flight on one GPU: while batch i is being decoded (the persistent decoder owns 96 of the 148 SMs at paper
    size and is latency-bound), batch i+1 is being encoded on the SMs the decoder leaves free -- its recurrences and, where they
    fit, its input-projection GEMMs too, otherwise the GEMMs between the decoder's segments (include/las_b200.h
    `las_pipeline_step`, csrc/fast_pipeline.cu).

        pipe = las.serve()
        for x in batches:                 # [B,T,F] device tensors
            out = pipe.submit(x)          # None for the first batch, then the previous batch's ServingResult
        last = pipe.flush()

    Every batch gets exactly what `las(x, None, 0, is_training=False)` returns for it (bit-identical: the decoder's segments carry
    its state on the device).  `x` must stay alive and unmodified until the next `submit` / `flush` has been enqueued behind it on
    the same stream (its listener runs inside that call's work).  Shapes or modes the concurrent schedule does not cover (fp32
    mode, variants, batches of more than 64 utterances) run the same two steps one after the other."""

    def __init__(self, las, want_attention=True):
        self.las = las
        self.want_attention = want_attention
        self._pending = None  # (enc, enc_lengths) of the batch encoded last and not decoded yet

    def _decode_call(self, enc, enc_lengths):
        sp = self.las.speller
        return sp._prepare_decode(enc, sp.max_label_len, enc_lengths=enc_lengths, want_attn=self.want_attention)

    def submit(self, x, input_lengths=None):
        las = self.las
        lis, sp = las.listener, las.speller
        _require_cuda(x, "input_x")
        holders = [getattr(lis, "pLSTM_layer" + str(i)).BLSTM for i in range(lis.num_layers)]
        mode = _mode_of(lis.precision)
        if mode != _mode_of(sp.precision):
            raise RuntimeError("the serving pipeline needs the listener and the speller in the same precision mode")
        with torch.cuda.device(x.device), lis._cache.enqueue_lock(x.device), sp._cache.enqueue_lock(x.device):
            lc = _prepare_listener(x, holders, lis.input_feature_dim, lis.hidden_size, mode, lis._cache, input_lengths, lis.cell,
                                   getattr(lis, "_is_replica", False))
            args = _cabi.PipelineArgs()
            args.x, args.x_lengths, args.listener_packed = lc.x.data_ptr(), (lc.lens.data_ptr() if lc.lens is not None else None), lc.packed.data_ptr()
            args.listener_dims = C.pointer(lc.dims)
            args.enc, args.enc_lengths = lc.enc.data_ptr(), (lc.enc_lens.data_ptr() if lc.enc_lens is not None else None)
            args.listener_ws, args.listener_ws_bytes = lc.ws.data_ptr(), lc.ws.numel()
            out = None
            if self._pending is not None:
                dc = self._decode_call(*self._pending)
                args.dec_io, args.speller_packed, args.speller_dims = C.pointer(dc.io), dc.packed.data_ptr(), C.pointer(dc.dims)
                args.steps, args.decode_mode, args.relu = dc.steps, dc.decode_mode, dc.relu
                args.speller_ws, args.speller_ws_bytes = dc.ws.data_ptr(), dc.ws.numel()
                out = ServingResult(dc.logp, dc.attn[:, 0] if dc.attn is not None and dc.attn.size(1) == 1 else dc.attn, dc.tokens)
            check(lc.lib.las_pipeline_step(C.byref(args), mode, lc.st))
            self._pending = (lc.enc, lc.enc_lens)
        return out

    def flush(self):
        """Decodes the batch submitted last; returns its ServingResult (None if nothing is pending)."""
        if self._pending is None:
            return None
        enc, enc_lens = self._pending
        self._pending = None
        sp = self.las.speller
        logp, attn, tokens = sp._decode(enc, sp.max_label_len, enc_lengths=enc_lens, want_attn=self.want_attention)
        return ServingResult(logp, attn[:, 0] if attn is not None and attn.size(1) == 1 else attn, tokens)


BeamSearchResult = collections.namedtuple("BeamSearchResult", ["tokens", "lengths", "scores", "token_logp"])
BeamSearchResult.__doc__ = """n-best hypotheses per utterance, best first (device tensors): tokens [B,N,S] int32 (<eos> after the end), lengths
[B,N] int32 (tokens up to and including the first <eos>, or S), scores [B,N] fp32 (sum of token_logp), token_logp [B,N,S] fp32 (0 after
the end)."""


BeamSearchAlignedResult = collections.namedtuple("BeamSearchAlignedResult", BeamSearchResult._fields + ("attention",))
BeamSearchAlignedResult.__doc__ = """BeamSearchResult's fields plus attention [B,N,S,U] fp32 ([B,N,S,heads,U] with multi_head > 1): the attention
weights the decoder computed at step t for the hypothesis row that token t was chosen from, 0 from lengths[b,n] on."""


def _check_beam_args(beam_width, nbest, length_penalty, steps, return_attention=False, early_exit=False):
    """The library's limits, checked on the host so that bad arguments fail before anything reaches the device."""
    for name, flag in (("return_attention", return_attention), ("early_exit", early_exit)):
        if not isinstance(flag, bool):
            raise ValueError(f"{name} must be a bool, got {flag!r}")
    if isinstance(beam_width, bool) or not isinstance(beam_width, int) or not 1 <= beam_width <= 32:
        raise ValueError(f"beam_width must be an int in [1, 32], got {beam_width!r}")
    if isinstance(nbest, bool) or not isinstance(nbest, int) or not 1 <= nbest <= beam_width:
        raise ValueError(f"nbest must be an int in [1, beam_width={beam_width}], got {nbest!r}")
    if isinstance(length_penalty, bool) or not isinstance(length_penalty, (int, float)) or not math.isfinite(length_penalty) \
            or length_penalty < 0:
        raise ValueError(f"length_penalty must be a finite number >= 0, got {length_penalty!r}")
    if isinstance(steps, bool) or not isinstance(steps, int) or steps < 1:
        raise ValueError(f"the number of decoder steps must be an int >= 1, got {steps!r}")


def _check_unit(rnn_unit, precision="fp32"):
    """-> "LSTM" | "GRU" | "RNN" (the reference resolves the string with getattr(nn, rnn_unit.upper()))."""
    unit = str(rnn_unit).upper()
    if unit not in _cabi.CELLS:
        raise NotImplementedError(f"rnn_unit={rnn_unit!r}: LSTM, GRU and RNN cells are implemented (SURVEY.md section 8 row f4)")
    return unit


class pBLSTMLayer(nn.Module):
    """model/las_model.py:66-91: halve the time axis by pairing frames, then a bidirectional LSTM."""

    def __init__(self, input_feature_dim, hidden_dim, rnn_unit="LSTM", dropout_rate=0.0, precision=None):
        super().__init__()
        self.precision = precision or _default_precision()
        self.cell = _check_unit(rnn_unit, self.precision)
        self.rnn_unit = getattr(nn, self.cell)  # the reference stores the class here (:69)
        self.input_feature_dim = input_feature_dim
        self.hidden_dim = hidden_dim
        # same parameter names as nn.LSTM(input_feature_dim*2, hidden_dim, 1, bidirectional=True) (:72-79)
        self.BLSTM = LSTMWeights(input_feature_dim * 2, hidden_dim, 1, bidirectional=True, cell=self.cell)
        self._cache = _Cache()

    def forward(self, input_x):
        out = _run_listener(input_x, [self.BLSTM], self.input_feature_dim, self.hidden_dim, _mode_of(self.precision), self._cache,
                            cell=self.cell, is_replica=getattr(self, "_is_replica", False))
        h = self.hidden_dim
        h_n = torch.stack([out[:, -1, :h], out[:, 0, h:]])  # final hidden of each direction
        return out, (h_n, None)


class Listener(nn.Module):
    """model/las_model.py:96-134: stack of `num_layers` pBLSTM layers, [B,T,F] -> [B, T/2^L, 2H]."""

    def __init__(self, input_feature_dim, hidden_size, num_layers, rnn_unit, use_gpu=True, dropout_rate=0.0, **kwargs):
        super().__init__()
        self.precision = kwargs.get("precision") or _default_precision()
        self.cell = _check_unit(rnn_unit, self.precision)
        self.input_feature_dim = input_feature_dim
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.rnn_unit = rnn_unit
        self.dropout_rate = dropout_rate
        assert self.num_layers >= 1, "Listener should have at least 1 layer"
        self.pLSTM_layer0 = pBLSTMLayer(input_feature_dim, hidden_size, rnn_unit=rnn_unit, dropout_rate=dropout_rate,
                                        precision=self.precision)
        for i in range(1, self.num_layers):
            setattr(self, "pLSTM_layer" + str(i), pBLSTMLayer(hidden_size * 2, hidden_size, rnn_unit=rnn_unit, dropout_rate=dropout_rate,
                                                              precision=self.precision))
        self._cache = _Cache()

    def forward(self, input_x, input_lengths=None):
        """`input_lengths=None` is the reference behaviour (padding is processed as data); with lengths the call returns
        (listener_feature, enc_lengths)."""
        holders = [getattr(self, "pLSTM_layer" + str(i)).BLSTM for i in range(self.num_layers)]
        return _run_listener(input_x, holders, self.input_feature_dim, self.hidden_size, _mode_of(self.precision), self._cache,
                             lengths=input_lengths, cell=self.cell, is_replica=getattr(self, "_is_replica", False))


class Attention(nn.Module):
    """model/las_model.py:249-318 (single head, 'dot')."""

    def __init__(self, mlp_preprocess_input, preprocess_mlp_dim, activate, mode="dot", input_feature_dim=512, multi_head=1):
        super().__init__()
        self.mode = mode.lower()
        self.mlp_preprocess_input = mlp_preprocess_input
        self.multi_head = multi_head
        self.input_feature_dim = input_feature_dim
        if multi_head < 1:
            raise ValueError(f"multi_head must be >= 1, got {multi_head}")
        if multi_head > 1 and not mlp_preprocess_input:
            raise ValueError("multi_head > 1 needs use_mlp_in_attention=True: the heads are slices of phi's output (model/las_model.py:303-305)")
        if self.mode != "dot":
            raise NotImplementedError("only 'dot' attention exists in the reference (model/las_model.py:315-317)")
        if mlp_preprocess_input:
            self.preprocess_mlp_dim = preprocess_mlp_dim
            self.phi = LinearWeights(input_feature_dim, preprocess_mlp_dim * multi_head)
            self.psi = LinearWeights(input_feature_dim, preprocess_mlp_dim)
            if self.multi_head > 1:  # model/las_model.py:268-269
                self.dim_reduce = LinearWeights(input_feature_dim * multi_head, input_feature_dim)
            if activate != "None":
                if activate != "relu":
                    raise NotImplementedError(f"mlp_activate_in_attention={activate!r}: only 'relu' and 'None' are implemented")
                self.activate = "relu"
            else:
                self.activate = None

    @property
    def relu_flag(self):
        return 1 if (self.mlp_preprocess_input and self.activate) else 0

    @property
    def mlp_dim(self):
        return self.preprocess_mlp_dim if self.mlp_preprocess_input else self.input_feature_dim

    def project_listener_feature(self, listener_feature):
        """psi(listener_feature) with activation -- the step-invariant half of :276-285, computed once."""
        enc = _f32c(listener_feature)
        if not self.mlp_preprocess_input:
            return enc
        _require_cuda(enc, "listener_feature")
        lib = _cabi.load_library()
        b, u, e = enc.shape
        d = self.preprocess_mlp_dim
        psi = torch.empty(b, u, d, dtype=torch.float32, device=enc.device)
        with torch.cuda.device(enc.device):
            w, bias = _f32c(self.psi.weight), _f32c(self.psi.bias)
            check(lib.las_psi_precompute(ptr(enc), ptr(w), ptr(bias), b, u, e, d, self.relu_flag, ptr(psi), current_stream_ptr(enc.device)))
        return psi

    def forward(self, decoder_state, listener_feature):
        _require_cuda(listener_feature, "listener_feature")
        lib = _cabi.load_library()
        enc = _f32c(listener_feature)
        state = _f32c(decoder_state).reshape(decoder_state.size(0), -1)
        b, u, e = enc.shape
        hs = state.size(1)
        psi = self.project_listener_feature(enc)
        nh = self.multi_head
        score = torch.empty(nh, b, u, dtype=torch.float32, device=enc.device)
        context = torch.empty(b, e, dtype=torch.float32, device=enc.device)
        with torch.cuda.device(enc.device):
            if self.mlp_preprocess_input:
                w, bias = _f32c(self.phi.weight), _f32c(self.phi.bias)
            else:
                w = bias = None
            wdr = bdr = None
            if nh > 1:
                wdr, bdr = _f32c(self.dim_reduce.weight), _f32c(self.dim_reduce.bias)
            check(lib.las_attention_forward(ptr(state), ptr(enc), ptr(psi), ptr(w), ptr(bias), b, u, e, hs, self.mlp_dim,
                                            self.relu_flag, nh, ptr(wdr), ptr(bdr), None, ptr(score), ptr(context),
                                            current_stream_ptr(enc.device)))
        return list(score.unbind(0)), context


class Speller(nn.Module):
    """model/las_model.py:138-238: attention decoder; the whole step loop runs on the device."""

    def __init__(self, vocab_size, hidden_size, rnn_unit, num_layers, max_label_len, use_mlp_in_attention,
                 mlp_dim_in_attention, mlp_activate_in_attention, listener_hidden_size, multi_head, decode_mode,
                 use_gpu=True, **kwargs):
        super().__init__()
        self.precision = kwargs.get("precision") or _default_precision()
        self.cell = _check_unit(rnn_unit, self.precision)
        self.rnn_unit = getattr(nn, self.cell)  # the reference stores the class (:156); serialize() writes it under "etype"
        self.hidden_size = hidden_size
        self.num_layers = num_layers
        self.max_label_len = max_label_len
        self.decode_mode = decode_mode
        self.use_gpu = use_gpu
        self.float_type = torch.cuda.FloatTensor if use_gpu else torch.FloatTensor
        self.label_dim = vocab_size
        if decode_mode not in (0, 1, 2):
            raise ValueError(f"decode_mode must be 0 (raw), 1 (greedy) or 2 (sample), got {decode_mode}")
        if hidden_size != 2 * listener_hidden_size:
            raise ValueError(
                f"hidden_size ({hidden_size}) must equal 2*listener_hidden_size ({2 * listener_hidden_size}): the rnn input is "
                "[one-hot || encoder feature] (model/las_model.py:165,198)"
            )
        self.rnn_layer = LSTMWeights(vocab_size + hidden_size, hidden_size, num_layers=num_layers, cell=self.cell)
        self.attention = Attention(
            mlp_preprocess_input=use_mlp_in_attention,
            preprocess_mlp_dim=mlp_dim_in_attention,
            activate=mlp_activate_in_attention,
            input_feature_dim=2 * listener_hidden_size,
            multi_head=multi_head,
        )
        self.character_distribution = LinearWeights(hidden_size * 2, vocab_size)
        self._cache = _Cache()

    # ---- device plumbing -------------------------------------------------------------------------------
    def _dims(self, b, u, e):
        at = self.attention
        return SpellerDims(b, u, e, self.hidden_size, self.num_layers, self.label_dim,
                           at.preprocess_mlp_dim if at.mlp_preprocess_input else 0, at.multi_head, 0 if at.mlp_preprocess_input else 1,
                           _cabi.CELLS[self.cell])

    def _packed(self, lib, dims, mode, device, st, beam=False):
        """Packed weights of the greedy decoder, or with `beam` those of beam search (las_speller_beam_pack), cached side by side."""
        tensors = _weight_tensors(self)
        for w in tensors:
            _require_cuda(w, "speller weight")
            if w.device != device:
                raise RuntimeError(f"speller weights are on {w.device}, listener_feature on {device}")
        slot = ("beam", mode) if beam else mode
        key = _Cache.tensors_key(tensors, slot)
        packed = self._cache.lookup(device, slot, key, getattr(self, "_is_replica", False))
        if packed is None:
            arr, keep = _lstm_weight_array(self.rnn_layer, self.num_layers, 1)
            at, cd = self.attention, self.character_distribution
            w = SpellerWeights()
            w.rnn_host = C.cast(arr, C.POINTER(LstmWeights))
            ts = [_f32c(t) for t in (cd.weight, cd.bias)]
            w.w_cd, w.b_cd = (t.data_ptr() for t in ts)
            if at.mlp_preprocess_input:
                ta = [_f32c(t) for t in (at.phi.weight, at.phi.bias, at.psi.weight, at.psi.bias)]
                w.w_phi, w.b_phi, w.w_psi, w.b_psi = (t.data_ptr() for t in ta)
                ts += ta
            if at.multi_head > 1:
                td = [_f32c(t) for t in (at.dim_reduce.weight, at.dim_reduce.bias)]
                w.w_dr, w.b_dr = (t.data_ptr() for t in td)
                ts += td
            size_fn, pack_fn = (lib.las_speller_beam_packed_bytes, lib.las_speller_beam_pack) if beam else \
                (lib.las_speller_packed_bytes, lib.las_speller_pack)
            nbytes = size_fn(C.byref(dims), mode)
            packed = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=device)
            check(pack_fn(C.byref(w), C.byref(dims), mode, ptr(packed), packed.numel(), st))
            self._cache.store(device, slot, key, packed)
            del keep, ts
        return packed

    def _prepare_decode(self, enc, steps, gt_dense=None, gt_index=None, state=None, word=None, context=None, enc_lengths=None,
                        want_attn=True, nll_labels=None, segment_steps=0, early_exit=False, eos_token=1):
        """Checks, packed weights, workspace, outputs and the las_decode_io of one decode call (the caller holds the enqueue lock)."""
        _require_cuda(enc, "listener_feature")
        lib = _cabi.load_library()
        enc = _f32c(enc)
        b, u, e = enc.shape
        mode = _mode_of(self.precision)
        dims = self._dims(b, u, e)
        dev = enc.device
        # the kernels index these with strides derived from (B, label_dim): a mismatching tensor must raise here, as the
        # reference does at torch.cat (model/las_model.py:236), not read out of bounds
        if e != self.hidden_size:
            raise RuntimeError(f"listener_feature has {e} features; the speller was built for {self.hidden_size} (model/las_model.py:165,198)")
        if gt_dense is not None and (gt_dense.dim() != 3 or gt_dense.size(0) != b or gt_dense.size(2) != self.label_dim or gt_dense.size(1) < steps):
            raise RuntimeError(f"ground_truth has shape {tuple(gt_dense.shape)}; expected [{b}, >={steps}, {self.label_dim}]")
        if gt_index is not None:
            if gt_index.dim() != 2 or gt_index.size(0) != b or gt_index.size(1) < steps:
                raise RuntimeError(f"ground_truth indices have shape {tuple(gt_index.shape)}; expected [{b}, >={steps}]")
        if enc_lengths is not None and enc_lengths.numel() != b:
            raise RuntimeError(f"enc_lengths has {enc_lengths.numel()} entries for a batch of {b}")
        if nll_labels is not None and (nll_labels.dim() != 2 or nll_labels.size(0) != b):
            raise RuntimeError(f"nll_labels has shape {tuple(nll_labels.shape)}; expected [{b}, S']")
        for name, t, shape in (("state h", state[0] if state is not None else None, (self.num_layers, b, self.hidden_size)),
                               ("word", word, (b, self.label_dim)), ("context", context, (b, e))):
            if t is not None and tuple(t.shape) != shape:
                raise RuntimeError(f"{name} has shape {tuple(t.shape)}; expected {shape}")
        st = current_stream_ptr(dev)
        packed = self._packed(lib, dims, mode, dev, st)
        ws_bytes = lib.las_speller_workspace_bytes(C.byref(dims), steps, mode)
        ws = self._cache.workspace(("speller", dev, mode, st.value), ws_bytes, dev)
        logp = torch.empty(steps, b, self.label_dim, dtype=torch.float32, device=dev)
        attn = torch.empty(steps, self.attention.multi_head, b, u, dtype=torch.float32, device=dev) if want_attn else None
        tokens = torch.empty(steps, b, dtype=torch.int32, device=dev)
        keep = [enc, gt_dense, gt_index, enc_lengths, state, word, context]
        io = DecodeIO()
        io.enc = enc.data_ptr()
        io.psi = None
        io.gt_steps = 0
        if gt_dense is not None:
            io.gt_dense = gt_dense.data_ptr()
            io.gt_steps = gt_dense.size(1)
        if gt_index is not None:
            io.gt_index = gt_index.data_ptr()
            io.gt_steps = gt_index.size(1)
        if enc_lengths is not None:
            io.enc_lengths = enc_lengths.data_ptr()
        if int(self.decode_mode) == 2 and gt_dense is None and gt_index is None:
            # one draw from torch's global generator seeds the device-side generator (reproducible under torch.manual_seed)
            io.sample_seed = int(torch.randint(0, 2 ** 62, (1,)).item())
        if state is not None:
            io.h_state = state[0].data_ptr()
            io.c_state = state[1].data_ptr() if state[1] is not None else None
        if word is not None:
            io.word, io.context = word.data_ptr(), context.data_ptr()
        nll_terms = None
        if nll_labels is not None:
            # fused NLLLoss(ignore_index=0) terms (solver/solver.py:62,70-77): [S,B], zero where the label is 0 / past the labels
            nll_labels = nll_labels.to(device=dev, dtype=torch.int32).contiguous()
            nll_terms = torch.empty(steps, b, dtype=torch.float32, device=dev)
            io.nll_labels, io.nll_steps, io.nll_terms = nll_labels.data_ptr(), nll_labels.size(1), nll_terms.data_ptr()
            keep.append(nll_labels)
        steps_done = None
        io.segment_steps = int(segment_steps)
        if early_exit:
            steps_done = torch.zeros(1, dtype=torch.int32, device=dev)
            io.early_exit, io.eos_token, io.steps_done = 1, int(eos_token), steps_done.data_ptr()
        io.logp = logp.data_ptr()
        io.attn = attn.data_ptr() if attn is not None else None
        io.tokens = tokens.data_ptr()
        return _Call(lib=lib, io=io, packed=packed, dims=dims, steps=steps, mode=mode, ws=ws, st=st, logp=logp, attn=attn, tokens=tokens,
                     nll_terms=nll_terms, steps_done=steps_done, keep=keep, relu=self.attention.relu_flag, decode_mode=int(self.decode_mode))

    def _decode(self, enc, steps, **kw):
        """Runs `steps` decoder steps.  Returns (logp [S,B,V], attn [S,heads,B,U] | None, tokens [S,B])."""
        _require_cuda(enc, "listener_feature")
        with torch.cuda.device(enc.device), self._cache.enqueue_lock(enc.device):
            c = self._prepare_decode(enc, steps, **kw)
            self.last_nll_terms = c.nll_terms
            self.last_steps_done = c.steps_done
            check(c.lib.las_speller_decode(C.byref(c.io), ptr(c.packed), C.byref(c.dims), steps, c.decode_mode, c.mode, c.relu, ptr(c.ws),
                                           c.ws.numel(), c.st))
        return c.logp, c.attn, c.tokens

    def beam_search(self, listener_feature, beam_width=8, nbest=1, length_penalty=0.0, enc_lengths=None, max_steps=None,
                    return_attention=False, early_exit=False):
        """Beam-search decoding on the device (extension; include/las_b200.h las_speller_beam_search has the exact semantics).
        Every utterance keeps `beam_width` hypotheses for `max_steps` (default max_label_len) steps; a hypothesis ends at <eos>
        (`self.eos_token`, default 1).  The `nbest` best by score / length**length_penalty are returned, best first, as a
        BeamSearchResult of device tensors.  Draws nothing from numpy's or torch's random generators.

        `return_attention=True` returns a BeamSearchAlignedResult: the same fields plus each hypothesis's attention record.
        `early_exit=True` stops issuing decoder steps once every hypothesis has ended, checked every `self.early_exit_every` (default
        32) steps; the outputs are bit-identical to a full run.  Each check waits on the stream for a 4-byte flag, so it cannot be
        captured into a CUDA graph.  The steps run are left in `self.last_steps_done` (device int32[1], overwritten by the next
        early-exit beam search).  It is independent of `self.early_exit`, which only governs greedy decoding."""
        steps = self.max_label_len if max_steps is None else max_steps
        _check_beam_args(beam_width, nbest, length_penalty, steps, return_attention, early_exit)
        eos = getattr(self, "eos_token", 1)
        if not 0 <= eos < self.label_dim:
            raise ValueError(f"eos_token {eos} is not in [0, {self.label_dim})")
        if listener_feature.dim() != 3 or listener_feature.size(2) != self.hidden_size:
            raise ValueError(f"listener_feature has shape {tuple(listener_feature.shape)}; expected [B, U, {self.hidden_size}]")
        b, u, e = listener_feature.shape
        if enc_lengths is not None and enc_lengths.numel() != b:
            raise ValueError(f"enc_lengths has {enc_lengths.numel()} entries for a batch of {b}")
        _require_cuda(listener_feature, "listener_feature")
        if early_exit and torch.cuda.is_current_stream_capturing():
            # (the library refuses it as well; raising here also keeps a first call's weight packing out of the graph)
            raise RuntimeError("beam search with early_exit waits on the stream for its stop flag and cannot be captured into a CUDA graph")
        lib = _cabi.load_library()
        dev = listener_feature.device
        mode = _mode_of(self.precision)
        with torch.cuda.device(dev), self._cache.enqueue_lock(dev):
            enc = _f32c(listener_feature)
            dims = self._dims(b, u, e)
            st = current_stream_ptr(dev)
            packed = self._packed(lib, dims, mode, dev, st, beam=True)
            ws_bytes = lib.las_speller_beam_workspace_bytes(C.byref(dims), steps, beam_width, mode)
            ws = self._cache.workspace(("beam", dev, mode, st.value), ws_bytes, dev)
            lens = None if enc_lengths is None else enc_lengths.to(device=dev, dtype=torch.int32).contiguous()
            out = BeamSearchResult(tokens=torch.empty(b, nbest, steps, dtype=torch.int32, device=dev),
                                   lengths=torch.empty(b, nbest, dtype=torch.int32, device=dev),
                                   scores=torch.empty(b, nbest, dtype=torch.float32, device=dev),
                                   token_logp=torch.empty(b, nbest, steps, dtype=torch.float32, device=dev))
            io = BeamIO()
            io.enc, io.enc_lengths = enc.data_ptr(), (lens.data_ptr() if lens is not None else None)
            io.beam, io.nbest, io.eos_token, io.length_penalty = beam_width, nbest, eos, float(length_penalty)
            io.tokens, io.token_logp, io.lengths, io.scores = (t.data_ptr() for t in (out.tokens, out.token_logp, out.lengths, out.scores))
            if return_attention:
                nh = self.attention.multi_head
                attn = torch.empty((b, nbest, steps, u) if nh == 1 else (b, nbest, steps, nh, u), dtype=torch.float32, device=dev)
                # las_beam_io.attn_work: [S, heads, B*K, U] fp32, then [B, N, S] int32
                work = self._cache.workspace(("beam_attn", dev, st.value), 4 * steps * (nh * b * beam_width * u + b * nbest), dev)
                io.attn, io.attn_work = attn.data_ptr(), work.data_ptr()
                out = BeamSearchAlignedResult(*out, attention=attn)
            if early_exit:
                steps_done = self._cache.workspace(("beam_steps_done", dev, st.value), 4, dev)[:4].view(torch.int32)
                io.early_exit, io.segment_steps, io.steps_done = 1, int(getattr(self, "early_exit_every", 32)), steps_done.data_ptr()
            check(lib.las_speller_beam_search(C.byref(io), ptr(packed), C.byref(dims), steps, mode, self.attention.relu_flag, ptr(ws),
                                              ws.numel(), st))
            if early_exit:
                self.last_steps_done = steps_done
        return out

    # ---- reference API ---------------------------------------------------------------------------------
    def forward_step(self, input_word, last_hidden_state, listener_feature):
        """One decoder step (model/las_model.py:178-184).  input_word [B,1,V+E]; last_hidden_state (h,c) or None."""
        b = input_word.size(0)
        v = self.label_dim
        flat = _f32c(input_word).reshape(b, -1)
        word = flat[:, :v].contiguous()
        context = flat[:, v:].contiguous()
        lstm = self.cell == "LSTM"
        if last_hidden_state is None:
            h = torch.zeros(self.num_layers, b, self.hidden_size, dtype=torch.float32, device=flat.device)
            c = torch.zeros_like(h) if lstm else None
        elif lstm:
            h, c = (_f32c(t).clone() for t in last_hidden_state)
        else:  # nn.GRU / nn.RNN carry a single hidden-state tensor
            h, c = _f32c(last_hidden_state).clone(), None
        logp, attn, _ = self._decode(listener_feature, 1, state=(h, c), word=word, context=context)
        return logp[0], ((h, c) if lstm else h), context, list(attn[0].unbind(0))

    def forward(self, listener_feature, ground_truth=None, teacher_force_rate=0.9, enc_lengths=None, nll_labels=None,
                early_exit=None):
        """`nll_labels` ([B,S'] label indices; extension) makes the decoder also emit the NLLLoss(ignore_index=0) terms of
        solver/solver.py:62,70-77 as `self.last_nll_terms` [S,B], so the loss needs no pass over the log-probabilities.
        `early_exit` (extension, default `self.early_exit` = False; SURVEY.md section 8 row f4): free-running decoding stops once every
        utterance has emitted <eos> (token 1, utils/functions.py:124-125), checked on the device every `self.early_exit_every` steps; the
        remaining steps are filled with <eos> tokens and zero log-probs, `self.last_steps_done` (device int32[1]) says how many ran.
        The reference always runs max_label_len steps (model/las_model.py:205-209), which stays the default."""
        if ground_truth is None:
            teacher_force_rate = 0
        # one draw from numpy's global RNG per call, exactly like the reference (:189)
        teacher_force = True if np.random.random_sample() < teacher_force_rate else False

        gt_dense = gt_index = None
        if (ground_truth is None) or (not teacher_force):
            max_step = self.max_label_len
        else:
            max_step = ground_truth.size()[1]
            if ground_truth.dim() == 2:
                # extension (SURVEY.md section 8 row f2): [B,S] label indices instead of the reference's [B,S,V] one-hot
                # tensor -- V times less host-to-device traffic; index v feeds one_hot(v), a negative index the zero vector
                if not ground_truth.is_cuda and ground_truth.numel() and int(ground_truth.max()) >= self.label_dim:
                    # (checked on host tensors only: a device tensor would cost a sync per call; there an index >= V feeds the zero vector)
                    raise RuntimeError(f"ground_truth index {int(ground_truth.max())} is out of range for a vocabulary of {self.label_dim}")
                gt_index = ground_truth.to(device=listener_feature.device, dtype=torch.int32).contiguous()
            else:
                # `.type(self.float_type)` in the reference (:217): the label tensor is consumed as dense floats
                gt_dense = ground_truth.to(device=listener_feature.device, dtype=torch.float32).contiguous()
        if enc_lengths is not None:
            enc_lengths = enc_lengths.to(device=listener_feature.device, dtype=torch.int32).contiguous()
        if early_exit is None:
            early_exit = getattr(self, "early_exit", False)
        early_exit = bool(early_exit) and gt_dense is None and gt_index is None  # teacher forcing decodes every label
        logp, attn, tokens = self._decode(listener_feature, max_step, gt_dense=gt_dense, gt_index=gt_index, enc_lengths=enc_lengths,
                                          nll_labels=nll_labels, early_exit=early_exit, eos_token=getattr(self, "eos_token", 1),
                                          segment_steps=getattr(self, "early_exit_every", 32) if early_exit else 0)
        self.last_tokens = tokens  # [S,B] int32 argmax per step (device); not part of the reference API
        self.last_logp = logp      # [S,B,V] the buffer raw_pred_seq's entries are views of
        raw_pred_seq = list(logp.unbind(0))
        attention_record = [list(a.unbind(0)) for a in attn.unbind(0)]  # per step: one [B,U] tensor per head (:214,:292,:299)
        return raw_pred_seq, attention_record
