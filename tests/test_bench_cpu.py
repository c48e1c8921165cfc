"""CPU: the host-side logic of bench.py that can run without a GPU — the two arms print the same `config`, the
reference arm's line has the contract's keys, and the N > 1 parity checker (gathered rank-major bitmap + summed counts
against the streaming oracle over all N x pods) accepts a correct result and rejects a wrong word, a wrong count and
stray padding bits."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.fixture()
def bench(monkeypatch):
    import bench as b
    monkeypatch.setattr(b, "PODS", 640)
    monkeypatch.setattr(b, "GPUS", 2)
    monkeypatch.setattr(b, "SAMPLES", 120)
    return b


def _sharded_result(b, world, window):
    """what world ranks would gather: shards are whole words, so rank-major words == the global bitmap, padded"""
    import gpu_pruner_b200 as g
    from oracle import oracle_c
    total = b.PODS * world
    ref = oracle_c.decide_synth(b.SEED + 16 * window, 0, total, b.GPUS, b.SAMPLES, use_elig=True, n_threads=2)
    sh = g.shard_pods(total, 0, world)
    words = np.zeros(sh.words_per_rank * world, np.uint32)
    words[: len(ref["decision_bits"])] = ref["decision_bits"]
    return words, [ref["n_series"], ref["n_candidates"], ref["n_decisions"]]


@pytest.mark.parametrize("world", [1, 2, 8])
def test_parity_checker_accepts_the_oracle_and_rejects_corruption(bench, world):
    first, c_first = _sharded_result(bench, world, 0)
    last, c_last = _sharded_result(bench, world, 3)
    out = bench.check_parity(world, first, c_first, last, c_last, 3)
    assert out["ok"] and out["pods_checked"] == bench.PODS * world
    bad = last.copy()
    bad[len(bad) // 2] ^= 0x10
    assert not bench.check_parity(world, first, c_first, bad, c_last, 3)["ok"]
    assert not bench.check_parity(world, first, [c_first[0], c_first[1], c_first[2] + 1], last, c_last, 3)["ok"]
    if world > 1:                                   # a stale word in the padding behind the last real pod
        pad = first.copy()
        pad[-1] |= 1 << 31
        if (bench.PODS * world + 31) // 32 < len(pad):
            assert not bench.check_parity(world, pad, c_first, last, c_last, 3)["ok"]
    # the wrong window for the last step must not pass either (catches a stale double buffer)
    assert not bench.check_parity(world, first, c_first, first, c_first, 3)["ok"]


def test_config_is_identical_in_both_arms_and_reference_line_has_the_contract_keys():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    import bench as b
    assert line["config"] == b.workload_config(1)            # what the CUDA arm prints at N = 1
    assert "kernel" not in line["config"] and "model" not in line["config"]
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == line["value"] and len(cb["repetitions_ms_per_step"]) >= 3
    assert abs(line["value"] - b.PODS * b.GPUS * b.SAMPLES / (line["ms_per_step"] * 1e-3)) / line["value"] < 1e-6


def test_dump_outputs_hold_the_last_timed_step(bench, tmp_path, monkeypatch, capsys):
    """--dump-outputs: the bitmap and counts of the LAST of the K timed steps (window (K - 1) % ROTATE), as float64"""
    import argparse
    from oracle import oracle_c
    monkeypatch.setattr(oracle_c, "pool_pin", lambda on=True: None)   # keep this process's oracle pool unpinned
    steps = 3
    args = argparse.Namespace(gpus=1, steps=steps, warmup=3, dump_outputs=str(tmp_path / "out"))
    assert bench.run_reference(args) == 0
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == steps
    bits, counts = np.load(tmp_path / "out" / "decision_bits.npy"), np.load(tmp_path / "out" / "counts.npy")
    assert bits.dtype == counts.dtype == np.float64
    ref = oracle_c.decide_synth(bench.SEED + 16 * ((steps - 1) % bench.ROTATE), 0, bench.PODS, bench.GPUS, bench.SAMPLES,
                                use_elig=True, n_threads=2)
    assert np.array_equal(bits, ref["decision_bits"].astype(np.float64))
    assert counts.tolist() == [ref["n_series"], ref["n_candidates"], ref["n_decisions"]]
    other = oracle_c.decide_synth(bench.SEED, 0, bench.PODS, bench.GPUS, bench.SAMPLES, use_elig=True, n_threads=2)
    assert not np.array_equal(other["decision_bits"], ref["decision_bits"])   # the window really tells the steps apart


def test_steps_below_one_are_refused():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert p.returncode == 2 and "--steps" in p.stderr


def test_cuda_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)
