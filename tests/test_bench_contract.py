"""The CPU arm of bench.py (`--impl reference`) prints the contract's JSON line: checked here with a tiny sample
(ANCE_BENCH_TINY_CPU) so that the CPU suite stays fast; the GPU arm is exercised by the driver on a B200."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, ANCE_BENCH_TINY_CPU="1", **extra_env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_json_line():
    lines = _run({})
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["higher_is_better"] is True and d["value"] > 0 and d["unit"] and d["metric"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["config"]["index_rows"] == 8841823 and d["config"]["topk"] == 200 and "workload" in d["config"]
    assert isinstance(base, dict)   # the metric string is free text; the config is what BASELINE.json's configs[1] names


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_dump_outputs_is_a_fixed_sample_in_float(tmp_path):
    """--dump-outputs: outputs land as <name>.npy in float32 / float64 (labels exact), larger ones as the same seeded
    sample of rows in every run, all of it within 64 MB at the default workload's sizes."""
    import numpy as np
    import torch

    import bench
    rng = np.random.default_rng(1)
    outputs = {"passage_emb": torch.from_numpy(rng.standard_normal((37888, 768), dtype=np.float32)),
               "query_emb": rng.standard_normal((2368, 768), dtype=np.float32),
               "topk_labels": rng.integers(0, 8841823, size=(2368, 200))}
    bench.dump_outputs(str(tmp_path / "a"), outputs)
    bench.dump_outputs(str(tmp_path / "b"), outputs)
    total = 0
    for name in outputs:
        a, b = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert np.array_equal(a, b) and a.shape[0] == min(bench.DUMP_MAX_ROWS, len(outputs[name]))
        total += a.nbytes
    assert np.load(tmp_path / "a" / "query_emb.npy").dtype == np.float32
    labels = np.load(tmp_path / "a" / "topk_labels.npy")
    assert labels.dtype == np.float64 and np.array_equal(labels, outputs["topk_labels"])
    P, rows = outputs["passage_emb"].numpy(), np.load(tmp_path / "a" / "passage_emb.npy")
    idx = np.searchsorted(np.sort(P[:, 0]), rows[:, 0])
    idx = np.argsort(P[:, 0])[idx]                      # the input row each dumped row came from
    assert np.array_equal(P[idx], rows) and (np.diff(idx) > 0).all()
    assert total <= 64 << 20
