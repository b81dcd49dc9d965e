"""CPU: bench.py's reference arm (the CPU port of the reference, the one place outside tests/
that may execute oracle/) prints exactly one JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    # the default headline workload is llama2-7B (27 GB of host weights for the CPU arm): the contract is
    # checked on stories15M through the documented override (synthetic weights unless the real checkpoint
    # is staged in assets/)
    env = dict(os.environ, L2B_BENCH_CPU_BUDGET_S="3", L2B_BENCH_WORKLOAD="stories15M")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, env=env, cwd=ROOT, timeout=300)
    assert r.returncode == 0, r.stderr[-1500:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["config"]["workload"] == "stories15M" and d["n_gpus"] == 1
    # same keys / values as the GPU arm's config, and the CLI's steps / warm-up echoed (VERDICT r1 #2)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.bench_config("stories15M", 256, 1)
    assert d["steps"] == 2 and d["warmup"] == 1
    assert 2 <= d["sampled_positions_per_step"] <= 256
    assert abs(d["ms_per_step"] - 1e3 * 256 / d["value"]) < 1e-6 * d["ms_per_step"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 10 and d["gpu_launches"] == 0


def test_gpu_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True,
                       text=True, cwd=ROOT, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)


def test_default_headline_workload_is_the_same_at_every_gpu_count():
    """SCALE divides the N-GPU value by the 1-GPU value: both must be the same workload."""
    sys.path.insert(0, ROOT)
    import argparse
    import bench
    os.environ.pop("L2B_BENCH_WORKLOAD", None)
    for n in (1, 2, 4, 8):
        assert bench.pick_workload(argparse.Namespace(workload="auto", gpus=n)) == "llama2-7B"


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, cwd=ROOT, timeout=300)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_step_outputs_sample_only_the_positions_that_ran():
    """A cache larger than KV_SAMPLE floats is reduced to the same seeded sample every time, drawn from
    the rows of the positions the step ran (values here encode layer, position and column)."""
    sys.path.insert(0, ROOT)
    import types
    import bench
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint((512, 1376, 8, 8, 8, 1000, 2048))
    L, S, kv, positions = ck.n_layers, ck.seq_len, ck.dim, 300
    cache = np.arange(L * S * kv, dtype=np.float64)
    t = types.SimpleNamespace(ck=ck, state=lambda name: np.ones(kv, np.float32) if name == "x" else cache)
    a = bench.step_outputs(t, positions, np.arange(positions, dtype=np.int32), False)
    b = bench.step_outputs(t, positions, np.arange(positions, dtype=np.int32), False)
    assert L * positions * kv > bench.KV_SAMPLE
    for name in ("key_cache", "value_cache"):
        assert a[name].size == bench.KV_SAMPLE and np.array_equal(a[name], b[name])
        pos = (a[name].astype(np.int64) // kv) % S
        assert pos.max() < positions and len(np.unique(pos)) == positions
        assert len(np.unique(a[name].astype(np.int64) // (S * kv))) == L
    assert a["tokens"].dtype == np.float64 and a["x"].size == kv


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs writes what the last timed l2b_generate_argmax call computed (last position's logits,
    final hidden state, key / value cache rows; token ids, here the forced input), identical to a direct
    run on the same seeded inputs; and --steps 2 times exactly two runs of the positions."""
    positions = 32
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "stories110M", "--also", "none",
                        "--no-cpu-baseline", "--steps", "2", "--warmup", "1", "--positions", str(positions),
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-1500:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    names = ("tokens", "logits", "x", "key_cache", "value_cache")
    assert sorted(os.listdir(tmp_path)) == sorted(f"stories110M_{n}.npy" for n in names)
    got = {n: np.load(tmp_path / f"stories110M_{n}.npy") for n in names}
    sys.path.insert(0, ROOT)
    import bench
    import llama2_zig_b200 as l2b
    from llama2_zig_b200.checkpoint import shape_checkpoint
    ck = shape_checkpoint("stories110M")
    forced = bench.teacher_tokens(positions + 1, ck.vocab_size)[1:]
    with l2b.Transformer(ck, synthetic_seed=bench.SYNTH_SEED["stories110M"]) as t:
        tokens = t.generate_argmax(1, 0, positions, forced=forced, stop_on_bos=False)
        _, launches_per_run = t.last_timing()
        want = {"tokens": tokens.astype(np.float64), "logits": t.state("logits"), "x": t.state("x")}
        for n in ("key_cache", "value_cache"):
            want[n] = t.state(n).reshape(ck.n_layers, ck.seq_len, -1)[:, :positions].ravel()
    for n in names:
        assert got[n].dtype == (np.float64 if n == "tokens" else np.float32), n
        assert np.array_equal(got[n], want[n]), n
    assert launches_per_run > positions and line["steps"] == 2 and line["gpu_launches"] == 2 * launches_per_run
