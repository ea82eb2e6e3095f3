#!/usr/bin/env python
"""bench.py -- LAS forward hot path on B200: audio-seconds per second (RTFx) + microseconds per decoder step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--precision bf16|fp16|fp32]
                    [--workload c3|c2|c4|c5|yaml] [--dump-outputs DIR]

A "step" is one pass of the hot path (Listener pBLSTM encoder + Speller greedy attention-decoder loop) over one
synthetic batch.  Workloads are BASELINE.json configs (SURVEY.md section 8):
    c3 (default, the one the metric is quoted on): paper LAS (256x3 / 512x2), batch 64 x 1600 frames, 300-char greedy
    c2: small LAS (128x2 / 256x2), batch 32 x 1600 frames, 300-char greedy
    c4: paper LAS long-form, batch 16 x 3000 frames, 600-char greedy
    yaml: the reference's shipped YAML size (listener 512x3, speller 1024x2, batch 16, 576 steps): 34 MB of decoder LSTM weights do
        not fit on chip, so the bf16 mode decodes on the generic tensor-core path (one tcgen05 GEMM per cell and step)
    c5: paper LAS, ONE global batch of 512 x 1600 frames sharded 512/N per GPU (strong scaling; N = 1/2/4 run the decoder in
        chunks of 64 utterances per persistent launch); the gathered shard tokens are compared with a single-GPU decode
N > 1 (torchrun, one rank per GPU): every rank runs the same per-GPU batch on its own shard of utterances (weak
scaling: 64 utterances per GPU = BASELINE.json config 5's 8-GPU point); there is no data-path collective, NCCL only
brackets the timed region and reduces the time (MAX) and a token checksum.

One JSON line on rank 0.  `value` = whole-job audio-s/s with inputs resident in HBM (CUDA events, max over ranks);
`e2e` = same through LAS.forward with pinned-host inputs copied in and the decoded tokens copied out every step;
`roofline` = dominant launch group against the measured peak; `cpu_baseline` = oracle/las_ref_torch.py (the
reference's torch op sequence) timed on this box's host cores on a bounded sample.
`--impl reference` times that CPU path alone (rank 0 only); `--impl reference-gpu` times the same op sequence on cuda:0
(torch -> cuDNN RNN / cuBLAS, the reference with use_gpu=True; SURVEY.md 2.1), which the default line also carries as
`gpu_baseline`.  `parity` compares this run's GPU token stream / log-probs with the CPU arm's on the same inputs.
`--dump-outputs DIR` writes what the timed path returned in its last timed step (tokens, log-probs, attention; c2 also
the teacher-forced loss) as DIR/<name>.npy in float32.  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    "c3": dict(cfg="paper", B=64, T=1600, S=300, desc="paper LAS (listener 256x3 pBLSTM, speller 512x2), batch 64 x 1600 frames, 300-char greedy decode"),
    "c2": dict(cfg="small", B=32, T=1600, S=300, desc="small LAS (listener 128x2, speller 256x2), batch 32 x 1600 frames, 300-char greedy decode"),
    "c4": dict(cfg="paper", B=16, T=3000, S=600, desc="paper LAS long-form, batch 16 x 3000 frames, 600-char greedy decode"),
    "yaml": dict(cfg="shipped", B=16, T=1600, S=576,
                 desc="the reference's shipped config/librispeech-config.yaml (listener 512x3, speller 1024x2, batch_size 16, max_label_len 576), "
                      "1600 frames, 576-char greedy decode"),
    "c5": dict(cfg="paper", B=512, T=1600, S=300, strong=True,
               desc="paper LAS, global batch 512 x 1600 frames sharded 512/N per GPU, 300-char greedy decode"),
}
FRAME_SEC = 0.01  # 10 ms frame hop (BASELINE.md: 3000 frames = 30 s)
DUMP_BYTES = 64_000_000


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tensor=d["bf16_tflops"], tensor_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tensor=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML polled every ~2 ms from a
    thread (nvidia-smi -lms is too coarse for a 30 ms region); falls back to nvidia-smi when pynvml is missing."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []
        self.sm, self.reasons, self.mx, self.stop_flag, self.thread, self.nvml = [], set(), None, False, None, None

    def _nvml_loop(self):
        n, h = self.nvml, self.handle
        bits = {"hw_slowdown": n.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown
                if hasattr(n, "nvmlClocksEventReasonHwThermalSlowdown") else 0x40,
                "sw_thermal_slowdown": n.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksThrottleReasonSwPowerCap}
        while not self.stop_flag:
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
                r = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, b in bits.items():
                    if r & b:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            import pynvml as n

            n.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = int(vis.split(",")[self.idx]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else self.idx
            self.handle = n.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
            self.nvml = n
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1)
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                    "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def dump_outputs(dirname, outs):
    """Writes each of `outs` (name -> tensor with the utterances on axis 1, or a scalar) as <dirname>/<name>.npy in float32.
    Above DUMP_BYTES in all, a fixed seeded sample of the utterances is kept (the same in every run), listed in
    utterance_index.npy."""
    import numpy as np

    arrs = {k: v.detach().float().cpu().numpy() for k, v in outs.items()}
    batch = max(a.shape[1] for a in arrs.values() if a.ndim > 1)
    if sum(a.nbytes for a in arrs.values()) > DUMP_BYTES:
        per_utt = sum(a.nbytes for a in arrs.values() if a.ndim > 1) / batch
        keep = np.sort(np.random.default_rng(0).choice(batch, int((DUMP_BYTES - (1 << 16)) // per_utt), replace=False))
        arrs = {k: (a[:, keep] if a.ndim > 1 else a) for k, a in arrs.items()}
        arrs["utterance_index"] = keep.astype(np.float32)
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(dirname, k + ".npy"), a)


def shared_config(args, wl, world):
    """`config` is the SAME dict in both arms (the driver compares them): it names the workload and says, per arm, what differs."""
    per_gpu = wl["B"] // world if wl.get("strong") else wl["B"]
    return {"workload": f"{args.workload}: {wl['desc']}", "per_gpu_batch": per_gpu, "frames": wl["T"], "decode_steps": wl["S"],
            "weights": "random init seed 17, 2-D params x3 (gain-3)",
            "precision": "ours: bf16 GEMM operands, fp32 accumulate / state / softmax (north_star bf16 mode) unless --precision fp32; "
                         "reference arm: fp32 on the host CPU",
            "l2": "ours: 256 MiB buffer written between timed steps (inside the timed region when the serving pipeline is on, untimed "
                  "otherwise); reference arm: host CPU, not applicable",
            "parallelism": "ours: one rank per GPU, utterance shards, no data-path collective; reference arm: rank 0, all host threads"}


def reference_arm(wl, sample_B, steps, warmup, device="cpu", seed=17, x=None):
    """The reference's op sequence (oracle/las_ref_torch.py) on the host cores (or, device="cuda", through torch/cuDNN on the
    GPU); returns (audio_s_per_s, info).  info["tokens"] / ["logp"] are the last run's greedy outputs, info["model"] the port."""
    import torch

    import las_testlib as tl
    from oracle.las_ref_torch import RefTorchLAS

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = tl.CONFIGS[wl["cfg"]]
    las = tl.build_model(wl["cfg"], max_label_len=wl["S"], seed=17, gain=3.0)
    m = RefTorchLAS(tl.state_dict_numpy(las), c["L"], c["sl"], device=device)
    if x is None:
        x, _ = tl.make_inputs(wl["B"], wl["T"], c["F"], wl["S"], c["V"], seed=seed)
    x = x[:sample_B]
    cuda = device != "cpu"
    if cuda:
        x = x.to(device)
    times, lis_t, logp = [], [], None
    for i in range(warmup + steps):
        if cuda:
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        enc = m.listener(x)
        if cuda:
            torch.cuda.synchronize()
        t1 = time.perf_counter()
        logp, attn = m.speller(enc, wl["S"], None, 1)
        if cuda:
            torch.cuda.synchronize()
        t2 = time.perf_counter()
        if i >= warmup:
            times.append(t2 - t0); lis_t.append(t1 - t0)
    tot = sum(times)
    audio = sample_B * wl["T"] * FRAME_SEC * len(times)
    info = dict(cores=torch.get_num_threads(), steps_run=len(times), warmup_run=warmup,
                sample=f"{sample_B} of the workload's {wl['B']} utterances x {wl['T']} frames, full {wl['S']}-step greedy decode, "
                f"{len(times)} timed runs after {warmup} warm-up", ms_per_step=1e3 * tot / len(times),
                listener_ms=1e3 * sum(lis_t) / len(times), us_per_decoder_step=1e6 * (tot - sum(lis_t)) / len(times) / wl["S"],
                model=m, enc=enc, logp=logp, attn=attn, tokens=logp.argmax(-1), c=c)
    return audio / tot, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--precision", default=None, choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-sample", type=int, default=0, help="utterances in the CPU-baseline sample (0 = the workload's batch, at most 64)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="time LAS.forward batch by batch instead of the cross-batch serving pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    strong = bool(wl.get("strong"))
    if strong and wl["B"] % world:
        raise SystemExit(f"workload {args.workload} shards {wl['B']} utterances: world size {world} must divide it")

    base = {"metric": "audio-sec/sec (RTFx)", "unit": "audio-s/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "data": "synthetic", "config": shared_config(args, wl, world)}
    cpu_sample = args.cpu_sample or min(wl["B"], 64)

    # ---------------------------------------------------------------- reference arms: rank 0 only
    if args.impl in ("reference", "reference-gpu"):
        if rank != 0:
            return
        on_gpu = args.impl == "reference-gpu"
        # one step = a whole 64-utterance batch through the reference's op sequence (1-20 s on the host cores): one warm-up step
        val, info = reference_arm(wl, cpu_sample, args.steps, min(args.warmup, 1), device="cuda:0" if on_gpu else "cpu")
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"tokens": info["tokens"], "logp": info["logp"], "attn": info["attn"]})
        out = dict(base, impl=args.impl, steps=info["steps_run"], warmup=info["warmup_run"], steps_requested=args.steps, value=val,
                   ms_per_step=info["ms_per_step"], dtype="f32",
                   cpu_baseline={"value": val, "unit": "audio-s/s", "cores": info["cores"], "kind": "port", "sample": info["sample"],
                                 "device": "cuda:0 (torch + cuDNN)" if on_gpu else "host CPU",
                                 "us_per_decoder_step": info["us_per_decoder_step"], "listener_ms": info["listener_ms"]},
                   e2e={"value": val, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, gpu_launches=0)
        print(json.dumps(out))
        return

    # ---------------------------------------------------------------- our arm
    # the contract is ONE JSON line on stdout: route fd 1 to stderr while libraries initialise (NCCL prints a banner there)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    import numpy as np
    import torch

    import las_testlib as tl
    from las_pytorch_b200 import _cabi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    lib = _cabi.load_library()
    if os.environ.get("LAS_PIPE_SPLIT"):  # A/B hook: decoder steps per pipeline segment, e.g. "160,92,48"
        for l, n in enumerate(os.environ["LAS_PIPE_SPLIT"].split(",")):
            lib.las_debug_set_option(20 + l, int(n))
    precision = args.precision or ("bf16" if lib.las_mode_available(_cabi.MODE_BF16) else "fp32")
    c = tl.CONFIGS[wl["cfg"]]
    T, S = wl["T"], wl["S"]
    B = wl["B"] // world if strong else wl["B"]  # utterances on this GPU
    las = tl.build_model(wl["cfg"], max_label_len=S, seed=17, gain=3.0, precision=precision).to(dev)
    if strong:  # one global batch (same seed on every rank), this rank's contiguous shard
        x_global, labels_global = tl.make_inputs(wl["B"], T, c["F"], S, c["V"], seed=17)
        x_host, labels = x_global[rank * B:(rank + 1) * B].clone(), labels_global[rank * B:(rank + 1) * B]
    else:       # each rank decodes its own utterances (different per rank, same shape)
        x_host, labels = tl.make_inputs(B, T, c["F"], S, c["V"], seed=17 + rank)
    x_host = x_host.pin_memory()
    x_dev = x_host.to(dev)
    labels_dev = labels.to(dev).to(torch.int32)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    tf_leg = args.workload == "c2"  # BASELINE.json config 2: "teacher-forced loss + greedy decode of 300 chars"
    use_pipeline = (not args.no_pipeline) and precision != "fp32" and hasattr(las, "serve") and not tf_leg and B <= 64

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(x):
        """One pass of the hot path over one batch: listener, (c2: teacher-forced decode with the fused NLL loss,) greedy decode."""
        enc = las.listener(x)
        if tf_leg:
            # c2: the teacher-forced decode (with the fused NLL loss) and the greedy decode read the same listener features and are
            # independent: they are issued on two streams and -- 32 LSTM + 32 attention CTAs each at the small model -- run
            # concurrently as two persistent kernels (LAS_BENCH_SERIAL_LEGS=1: one after the other on the caller's stream)
            cur = torch.cuda.current_stream(dev)
            serial = bool(os.environ.get("LAS_BENCH_SERIAL_LEGS"))
            if not serial:
                one_step.fork.record(cur)
                one_step.side.wait_event(one_step.fork)
            with torch.cuda.stream(cur if serial else one_step.side):
                np.random.seed(0)
                las.speller(enc, labels_dev, 1.1, nll_labels=labels_dev)
                one_step.loss = las.speller.last_nll_terms.sum() / float(labels_dev.numel())
                if not serial:
                    one_step.join.record(one_step.side)
            one_step.result = las.speller(enc, None, 0.0)
            if not serial:
                cur.wait_event(one_step.join)
                enc.record_stream(one_step.side)
            return las.speller.last_tokens
        one_step.result = las.speller(enc, None, 0.0)
        return las.speller.last_tokens

    one_step.side, one_step.fork, one_step.join = torch.cuda.Stream(device=dev), torch.cuda.Event(), torch.cuda.Event()

    if not tf_leg and not use_pipeline:
        def one_step(x):  # noqa: F811 -- plain LAS.forward (batches beyond one decoder launch group are chunk-pipelined inside it)
            one_step.result = las(x, None, 0.0, is_training=False)
            return las.speller.last_tokens

    pipe = las.serve() if use_pipeline else None

    def timed_step(x):
        """What the timed loop calls: through the serving pipeline the call returns the PREVIOUS batch's outputs (None first)."""
        if pipe is None:
            return one_step(x)
        out = timed_step.result = pipe.submit(x)
        return None if out is None else out.tokens

    for _ in range(args.warmup):
        timed_step(x_dev)
    # (the serving pipeline stays primed: the last warm-up batch is encoded and waits for its decoder, so that each of the K
    # timed submissions below does one full listener AND one full decode -- K batches' worth of work inside the timed region)
    barrier()

    # ---- timed region 1: device-resident inputs, CUDA events around the K steps, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    if not os.environ.get("LAS_BENCH_NOSAMPLER"):
        sampler.start()
    # one more untimed step with the clock sampler already polling NVML (its first queries stall the first step enqueued after
    # them by several ms: measured 8-16 ms on the first timed step, 4.18 ms on every later one), then the counters start
    timed_step(x_dev)
    barrier()
    if not os.environ.get("LAS_BENCH_NOPROF"):
        lib.las_prof_enable(2 if os.environ.get("LAS_BENCH_DEBUG") else 1)
    lib.las_launch_count(1)
    tokens = None
    if pipe is None:
        evs = []
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            tokens = one_step(x_dev)
            e1.record()
            evs.append((e0, e1))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        step_ms = [round(a.elapsed_time(b), 4) for a, b in evs]
    else:
        # the pipeline keeps two batches in flight (batch i+1's listener under batch i's decoder), so steps cannot be bracketed one
        # by one: one event pair around exactly K submissions in steady state (each = the listener of one batch + the decoder of the
        # batch before it; the pipeline was primed by the warm-up and is drained after the region).  The 256 MiB L2-flush writes
        # (one per step, ~0.07 ms each) are INSIDE this region.
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
        flush.zero_()  # the flush in front of the first timed step is outside the region (it absorbs the memory system's wake-up after
        e0.record()    # the barrier: 4-10 ms for this one 256 MiB write against 0.07 ms for each later one); the K-1 others are inside
        host_ms = []
        for i in range(args.steps):
            if i:
                flush.zero_()
            h0 = time.perf_counter()
            tokens = timed_step(x_dev)
            host_ms.append(round(1e3 * (time.perf_counter() - h0), 3))
            marks[i].record()
        e1.record()
        torch.cuda.synchronize()
        launches = int(lib.las_launch_count(0))
        ctypes_buf = ctypes.create_string_buffer(1 << 20)
        _cabi.check(lib.las_prof_report(ctypes_buf, len(ctypes_buf)))  # the K timed steps' launch groups, before the drain adds its own
        lib.las_prof_enable(0)
        pipe.flush()
        barrier()
        ms = e0.elapsed_time(e1)
        step_ms = [round(a.elapsed_time(b), 4) for a, b in zip([e0] + marks[:-1], marks)]
        base["host_enqueue_ms_each_step"] = host_ms
    clocks = sampler.stop()
    if pipe is None:
        launches = int(lib.las_launch_count(0))
        ctypes_buf = ctypes.create_string_buffer(1 << 20)
        _cabi.check(lib.las_prof_report(ctypes_buf, len(ctypes_buf)))
        lib.las_prof_enable(0)
    # what the last timed step returned (device tensors; the untimed passes below produce new ones); one attention head
    if pipe is None:
        preds, attns = one_step.result
        final = {"tokens": tokens, "logp": torch.stack(preds), "attn": torch.stack([a[0] for a in attns])}
        if tf_leg:
            final["teacher_forced_loss"] = one_step.loss
    else:
        r = timed_step.result
        final = {"tokens": r.tokens, "logp": r.logp, "attn": r.attn}
    groups = {}
    if os.environ.get("LAS_BENCH_DEBUG"):
        sys.stderr.write("PROF-RAW\n" + ctypes_buf.value.decode() + "\n")
    for line in ctypes_buf.value.decode().splitlines():
        name, t, n = line.rsplit(" ", 2)
        name = name.split("@")[0]
        g = groups.setdefault(name, [0.0, 0])
        g[0] += float(t); g[1] += int(n)
    # untimed extra passes with the listener's GEMM / recurrence overlap switched off (las_debug_set_option(6, 0)): the duration
    # of each input-projection GEMM running ALONE on the whole chip, which is what its roofline line is quoted on (against the
    # BURST tensor peak, as for any kernel timed in isolation).  Pass 1 uses the epilogue the pipeline runs (row-per-thread stores,
    # option 8 = 1: the variant that runs next to the recurrence); pass 2 the shared-memory-staged TMA-store epilogue a stand-alone
    # launch picks (reported alongside).
    alone, alone_tma = {}, {}
    if rank == 0:
        for store_opt, dst in ((1, alone), (0, alone_tma)):
            lib.las_debug_set_option(6, 0)
            lib.las_debug_set_option(8, store_opt)
            one_step(x_dev)
            torch.cuda.synchronize()
            lib.las_prof_enable(1)
            for _ in range(3):
                flush.zero_()
                one_step(x_dev)
            torch.cuda.synchronize()
            _cabi.check(lib.las_prof_report(ctypes_buf, len(ctypes_buf)))
            lib.las_prof_enable(0)
            lib.las_debug_set_option(6, 1)
            lib.las_debug_set_option(8, 0)
            for line in ctypes_buf.value.decode().splitlines():
                name, t, n = line.rsplit(" ", 2)
                dst[name] = dst.get(name, 0.0) + float(t) / 3
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    chk = torch.tensor([float(tokens.sum())], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(chk, op=dist.ReduceOp.SUM)  # the only data NCCL moves: a scalar checksum of the decoded tokens
    ms = float(t_ms)
    audio_per_step = world * B * T * FRAME_SEC
    value = audio_per_step * args.steps / (ms / 1e3)

    # ---- strong scaling (c5): the shards' tokens, gathered, must be the tokens one GPU decodes for the whole global batch
    shard_check = None
    if strong:
        gathered = None
        if dist is not None:
            gathered = [torch.empty_like(tokens) for _ in range(world)] if rank == 0 else None
            dist.gather(tokens.contiguous(), gathered, dst=0)
        if rank == 0:
            all_tok = torch.cat(gathered, dim=1) if gathered is not None else tokens
            las.listener(x_global[:2].to(dev))  # (first-use allocations for the other batch size stay out of the comparison run)
            enc_g = las.listener(x_global.to(dev))
            las.speller(enc_g, None, 0.0)
            single = las.speller.last_tokens
            shard_check = {"compared": "tokens of the N shards gathered on rank 0 vs one GPU decoding all 512 utterances",
                           "tokens_equal_fraction": float((all_tok == single).float().mean()),
                           "utterances_identical": int((all_tok == single).all(0).sum()), "utterances": int(single.size(1))}
            del enc_g
        if dist is not None:
            dist.barrier()

    # ---- timed region 2 (e2e): through the public API (LAS.forward / LAS.serve), pinned-host input copied in, decoded tokens
    # AND log-probabilities copied out, every step.  Double-buffered: step i+1's input is copied in on a copy stream while step i
    # computes, step i's results leave on the copy stream and are read on the host once their event fires (one step later).  Every
    # step's H2D and D2H are inside the timed wall-clock region; the closing barrier waits for the last of them.
    tok_host = [torch.empty(S, B, dtype=torch.int32).pin_memory() for _ in range(2)]
    logp_host = [torch.empty(S, B, c["V"], dtype=torch.float32).pin_memory() for _ in range(2)]
    xd = [torch.empty_like(x_dev) for _ in range(3)]
    copy_stream = torch.cuda.Stream(device=dev)
    out_stream = torch.cuda.Stream(device=dev)
    in_ready = [torch.cuda.Event() for _ in range(3)]
    in_free = [torch.cuda.Event() for _ in range(3)]
    res_ready = [torch.cuda.Event() for _ in range(2)]
    out_done = [torch.cuda.Event() for _ in range(2)]
    main = torch.cuda.current_stream(dev)
    host_checksum = 0

    def api_step(x):
        """-> (tokens [S,B] int32, logp [S,B,V]) of a finished batch on the device, or None (pipeline still filling)."""
        if tf_leg:  # c2: the same two decodes per batch as the device-timed step (listener once, TF + loss, greedy)
            one_step(x)
            return las.speller.last_tokens, las.speller.last_logp
        if pipe is None:
            preds, _ = las(x, None, 0.0, is_training=False)
            return las.speller.last_tokens, las.speller.last_logp
        o = pipe.submit(x)
        return None if o is None else (o.tokens, o.logp)

    def ship(res, k):
        """Device results -> pinned host buffers k on the output stream."""
        res_ready[k].record(main)
        with torch.cuda.stream(out_stream):
            out_stream.wait_event(res_ready[k])
            tok_host[k].copy_(res[0], non_blocking=True)
            logp_host[k].copy_(res[1], non_blocking=True)
            out_done[k].record(out_stream)

    for _ in range(min(args.warmup, 3)):  # untimed warm-up of exactly this path: first-use allocations; leaves the pipeline primed
        xd[2].copy_(x_host, non_blocking=True)
        r = api_step(xd[2])
        if r is not None:
            ship(r, 0)
    barrier()
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    with torch.cuda.stream(copy_stream):
        xd[0].copy_(x_host, non_blocking=True)
        in_ready[0].record(copy_stream)
    shipped = 0
    for i in range(args.steps):
        cur, nxt = i % 3, (i + 1) % 3
        if i + 1 < args.steps:
            with torch.cuda.stream(copy_stream):
                if i >= 2:
                    copy_stream.wait_event(in_free[nxt])  # the step that last read this buffer has finished with it
                xd[nxt].copy_(x_host, non_blocking=True)
                in_ready[nxt].record(copy_stream)
        main.wait_event(in_ready[cur])
        if i:
            flush.zero_()  # cold L2 for every step here too; the 256 MiB write (~0.07 ms) is inside this wall-clock region
        r = api_step(xd[cur])
        # (pipeline: batch i's input buffer is read by its listener during THIS call's enqueued work; it is reused 3 steps later)
        in_free[cur].record(main)
        if r is not None:
            if shipped >= 2:
                out_done[shipped & 1].synchronize()  # the results shipped two batches ago are on the host: buffer free again
                host_checksum += int(tok_host[shipped & 1][0, 0])
            ship(r, shipped & 1)
            shipped += 1
    for k in range(2):
        out_done[k].synchronize()
    host_checksum += int(tok_host[(shipped - 1) & 1][0, 0])
    barrier()
    e2e_s = time.perf_counter() - t0
    assert shipped == args.steps, (shipped, args.steps)
    if pipe is not None:
        pipe.flush()
    t_e2e = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = audio_per_step * args.steps / float(t_e2e)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, final)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- rooflines per launch group (per step averages; algorithmic work from SURVEY.md 8d); `roofline` = the dominant one
    peaks = measured_peaks()
    H, L, E, Hs, V, D, sl, U = c["H"], c["L"], 2 * c["H"], 2 * c["H"], c["V"], c["D"], c["sl"], T >> c["L"]
    per_step = {k: v[0] / args.steps for k, v in groups.items()}
    n_dec = 2 if tf_leg else 1  # decoder launches of S steps per timed step
    # a GEMM that runs concurrently with its layer's recurrence (on the SMs the recurrence leaves free) adds nothing to the step
    lis_ms = sum(v for k, v in per_step.items() if k.startswith("listener") and not k.endswith(".overlapped"))
    spl_ms = sum(v for k, v in per_step.items() if k.startswith("speller"))
    esize = 2 if precision != "fp32" else 4
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")  # dram bytes per launch from `ncu --set full` (tools/ncu_traffic.py)
    if os.path.exists(tp):
        traffic = json.load(open(tp)).get(f"{args.workload}:{precision}", {})

    def roof(name):
        dt = per_step[name] / 1e3
        extra = {}
        in_pipeline = True
        if name.endswith(".overlapped"):
            # quoted on the kernel running alone on the whole chip (untimed extra pass); the in-pipeline duration is kept alongside
            extra = {"ms_in_pipeline_overlapped_with_recurrence": per_step[name],
                     "epilogue": "row-per-thread stores (the variant that runs next to the recurrence)",
                     "timed": "alone on the chip in an untimed extra pass -> burst tensor peak"}
            name = name[: -len(".overlapped")]
            if name not in alone:
                return None
            dt = alone[name] / 1e3
            in_pipeline = False
            if name in alone_tma:
                extra["ms_alone_with_tma_store_epilogue"] = alone_tma[name]
        if dt <= 0:
            return None
        if name.endswith("input_gemm"):
            l = int(name.split(".")[1][1:])
            M, K = B * (T >> (l + 1)), (2 * c["F"] if l == 0 else 4 * H)
            fl, by = 2.0 * M * K * 8 * H, esize * M * K + esize * 8 * H * K + 4.0 * M * 8 * H
            if l == 0 or precision == "fp32":  # K = 2F: arithmetic intensity below the ridge -> bound by the fp32 output write
                r = {"bound": "hbm", "achieved": by / dt / 1e9, "peak": peaks["hbm"], "unit": "GB/s", "tflops": fl / dt / 1e12}
            else:  # isolated launch -> burst peak; a launch timed inside the step -> sustained peak
                r = {"bound": "tensor", "achieved": fl / dt / 1e12, "peak": peaks["tensor_sustained"] if in_pipeline else peaks["tensor"],
                     "unit": "TFLOP/s", "peak_kind": "sustained" if in_pipeline else "burst"}
        elif name == "speller.steps":
            by = n_dec * S * (B * U * (D + E) * esize + 4.0 * B * U + 4.0 * B * V)  # K + enc read once per step, attn + logp written
            r = {"bound": "hbm", "achieved": by / dt / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
                 "us_per_decoder_step": per_step[name] * 1e3 / (n_dec * S * max(1, -(-B // 64)))}
        elif name.endswith("recurrence"):  # serial chain: report the bytes it must move (P read + h written) against HBM, and us / serial step
            l = int(name.split(".")[1][1:])
            Tl = T >> (l + 1)
            by = B * Tl * (8 * H * 4.0 + 2 * H * 4.0)
            if l == 0 and precision != "fp32" and (2 * c["F"]) % 16 == 0:  # fused input projection: x_t (bf16) read instead of P
                by = B * Tl * (2 * c["F"] * 2.0 + 2 * H * 2.0)
            r = {"bound": "hbm", "achieved": by / dt / 1e9, "peak": peaks["hbm"], "unit": "GB/s", "us_per_serial_step": per_step[name] * 1e3 / Tl}
        elif name == "speller.psi":
            by = n_dec * (B * U * (E * 4.0 + D * 4.0) + D * E * 4.0)
            r = {"bound": "hbm", "achieved": by / dt / 1e9, "peak": peaks["hbm"], "unit": "GB/s"}
        else:
            return None
        r = dict({"kernel": name}, **r)
        r["frac"] = r["achieved"] / r["peak"]
        r["traffic"] = traffic.get(name)
        r["peak_source"] = peaks["source"]
        r["ms_per_launch_group"] = dt * 1e3
        r.update(extra)
        return r

    rooflines = [r for r in (roof(k) for k in sorted(per_step, key=per_step.get, reverse=True)) if r]
    roofline = rooflines[0] if rooflines else None

    out = dict(base, value=value, ms_per_step=ms / args.steps, dtype={"bf16": "bf16", "fp16": "f16", "fp32": "f32"}[precision],
               precision=precision, world=world,
               mode=("serving pipeline (LAS.serve): batch i+1's listener runs under batch i's decoder; K steady-state submissions (each = one "
                     "batch's listener + the previous batch's decoder) timed with one CUDA-event pair, L2-flush writes included")
               if pipe is not None else "LAS.forward batch by batch, CUDA events per step",
               ms_each_step=step_ms, us_per_decoder_step=1e3 * spl_ms / (n_dec * S * max(1, -(-B // 64))), listener_ms=lis_ms, speller_ms=spl_ms, phase_ms=per_step,
               clocks=clocks, gpu_launches=launches,
               e2e={"value": e2e_value, "unit": "audio-s/s", "h2d_bytes_per_step": x_host.numel() * 4,
                    "d2h_bytes_per_step": tok_host[0].numel() * 4 + logp_host[0].numel() * 4,
                    "d2h": "decoded tokens [S,B] int32 AND log-probabilities [S,B,V] fp32 (the reference API's return value); the attention "
                           "record stays on the device",
                    "pipeline": "H2D of step i+1 on a copy stream during step i, D2H on an output stream read event-synchronised later; "
                                "wall clock, L2 flush write included"},
               roofline=roofline, rooflines=rooflines, token_checksum=float(chk))
    if tf_leg:
        out["teacher_forced_loss"] = float(one_step.loss)
    if shard_check is not None:
        out["shard_check"] = shard_check
    if world == 1 and not args.no_cpu_baseline:
        # the reference's op sequence on this box's host cores, same weights and the same utterances: baseline AND parity checker
        v, info = reference_arm(wl, cpu_sample, 5 if cpu_sample * S <= 64 * 300 else 2, 1, x=x_host if not strong else x_global)
        out["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": info["cores"], "kind": "port", "sample": info["sample"],
                               "us_per_decoder_step": info["us_per_decoder_step"], "listener_ms": info["listener_ms"]}
        # parity of THIS run's outputs (the timed e2e path's last batch, as read back on the host) with the CPU arm's
        k = (shipped - 1) & 1
        ours_tok = tok_host[k][:, :cpu_sample].numpy()
        ours_logp = logp_host[k][:, :cpu_sample].numpy()
        ref_tok = info["tokens"].numpy()
        onehot = tl.onehot(torch.from_numpy(ours_tok.T.astype(np.int64)), c["V"])
        rescored, _ = info["model"].speller(info["enc"], S, onehot, 1)  # the reference, teacher-forced on OUR tokens
        same = (ours_tok == ref_tok)
        # calibration for the bf16 mode: the reference's own op sequence with only its 2-D weights rounded to bf16 vs itself
        # (free-running greedy decoding at these weights is chaotic: one near-tie flip changes the rest of an utterance)
        from oracle.las_ref_torch import RefTorchLAS

        rdt = torch.float16 if precision == "fp16" else torch.bfloat16
        sd_b = {k: (v.detach().cpu().to(rdt).float().numpy() if v.dim() == 2 else v.detach().cpu().numpy()) for k, v in las.state_dict().items()}
        mb = RefTorchLAS(sd_b, c["L"], c["sl"])
        xs = (x_host if not strong else x_global)[:cpu_sample]
        lb, _ = mb.speller(mb.listener(xs), S, None, 1)
        cal = float((lb.argmax(-1).numpy() == ref_tok).mean())
        out["parity"] = {"against": "cpu_baseline (oracle/las_ref_torch.py, fp32) on the same utterances and weights",
                         "utterances": cpu_sample, "token_agreement": float(same.mean()),
                         "utterances_identical": int(same.all(0).sum()),
                         "logp_max_abs": float(np.abs(ours_logp - rescored.numpy()).max()),
                         "logp_max_abs_is": "our greedy log-probs vs the reference teacher-forced on the tokens we fed back (every step)",
                         "logp_max_abs_free_running": float(np.abs(ours_logp - info["logp"].numpy()).max()),
                         "reference_with_bf16_rounded_weights_token_agreement" if precision != "fp16" else "reference_with_fp16_rounded_weights_token_agreement": cal}
    if world == 1 and not args.no_gpu_baseline:
        try:  # SURVEY.md 2.1: the reference's own op sequence with use_gpu=True on this B200 (torch -> cuDNN / cuBLAS), bounded
            v, info = reference_arm(wl, cpu_sample, 2, 1, device=str(dev), x=x_host if not strong else x_global)
            out["gpu_baseline"] = {"value": v, "unit": "audio-s/s", "kind": "port on cuda (torch + cuDNN, fp32; TF32 as torch defaults)",
                                   "sample": info["sample"], "ms_per_step": info["ms_per_step"],
                                   "us_per_decoder_step": info["us_per_decoder_step"], "listener_ms": info["listener_ms"]}
        except Exception as e:  # noqa: BLE001 -- a baseline must not take the bench line down
            out["gpu_baseline"] = {"unavailable": repr(e)[:200]}
    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    print(json.dumps(out), flush=True)
    if dist is not None:
        os.dup2(2, 1)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
