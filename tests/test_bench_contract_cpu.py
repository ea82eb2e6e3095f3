"""bench.py's reference arm (the CPU leg the driver launches as `bench.py --impl reference`) on a one-utterance sample:
one JSON line with the contract's keys, no GPU needed; under torchrun only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(extra_env=None, steps=1, extra_args=()):
    env = dict(os.environ, **(extra_env or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2", "--cpu-sample", "1",
                        "--steps", str(steps), "--warmup", "1", *extra_args], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = run_bench()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("audio-sec/sec") and d["unit"] == "audio-s/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "utterances" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("c2:")
    # the line reports the steps it ran and keeps the request alongside
    assert d["steps"] == 1 and d["steps_requested"] == 1 and "1 timed runs" in cb["sample"]
    # both arms print the same `config` dict (the driver compares them)
    sys.path.insert(0, ROOT)
    import argparse

    import bench

    ours = bench.shared_config(argparse.Namespace(workload="c2"), bench.WORKLOADS["c2"], 1)
    assert d["config"] == ours


def test_reference_arm_is_silent_on_other_ranks():
    assert run_bench({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_steps_and_dump_outputs(tmp_path):
    """--steps sets the number of timed steps; --dump-outputs writes the last step's outputs as float32 .npy files, the same
    in every run (seeded inputs and weights)."""
    import numpy as np

    dumps = []
    for i in range(2):
        d = json.loads(run_bench(steps=2, extra_args=("--dump-outputs", str(tmp_path / str(i))))[0])
        assert d["steps"] == 2 and "2 timed runs" in d["cpu_baseline"]["sample"]
        dumps.append({f[:-4]: np.load(tmp_path / str(i) / f) for f in os.listdir(tmp_path / str(i))})
    assert sorted(dumps[0]) == ["attn", "logp", "tokens"]
    S, V, U = 300, 30, 1600 >> 2  # workload c2: 300 decoder steps, 30 labels, 2 pyramid layers; one utterance
    assert dumps[0]["tokens"].shape == (S, 1) and dumps[0]["logp"].shape == (S, 1, V) and dumps[0]["attn"].shape == (S, 1, U)
    for name, a in dumps[0].items():
        assert a.dtype == np.float32
        assert np.array_equal(a, dumps[1][name]), name
    assert np.array_equal(dumps[0]["tokens"], dumps[0]["logp"].argmax(-1))


def test_dump_outputs_samples_utterances_above_the_size_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", (1 << 16) + 40 * 1000 * 4)  # room for 40 utterances of 1000 floats
    logp = torch.arange(64 * 1000, dtype=torch.float32).reshape(1, 64, 1000)
    outs = {"logp": logp, "loss": torch.tensor(1.5, dtype=torch.float64)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), outs)
    idx = np.load(tmp_path / "a" / "utterance_index.npy").astype(np.int64)
    assert len(idx) == 40 and np.array_equal(idx, np.unique(idx))
    assert np.array_equal(np.load(tmp_path / "a" / "logp.npy"), logp[:, idx].numpy())
    assert np.load(tmp_path / "a" / "loss.npy") == np.float32(1.5)
    for f in os.listdir(tmp_path / "a"):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
