"""bench.py end to end on a CPU box: the corpus generator, query decoding, recall, self-parity, oracle parity, CPU
baseline, roofline bookkeeping and the JSON contract, with the CPU oracle standing in for the GPU library
(tests/fake_plaid.py) on a tiny corpus.  Both arms.  The numbers mean nothing; the keys, types and the parity
verdicts do."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--docs-total", "3000", "--doclen", "24", "--log2k", "8", "--batch", "4", "--nq", "8", "--top-k", "5",
         "--n-full-scores", "64", "--recall-queries", "6", "--parity-queries", "5", "--docs-per-topic", "100",
         "--pool", "16", "--steps", "3", "--warmup", "1", "--threads", "2"]


def _run(extra):
    env = dict(os.environ, PB_BENCH_LIB="fake_plaid", PB_BENCH_DEVICE="cpu", PB_BENCH_CHUNK_DOCS="1000",
               PYTHONPATH=os.path.join(ROOT, "tests") + os.pathsep + ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL + extra, env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_b200_arm_contract_on_the_cpu_stand_in():
    d = _run([])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert "workload" in d["config"] and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    # the stand-in IS the oracle: parity and self-parity must be perfect, recall is a number in [0, 1]
    assert d["parity"]["ids_identical"] == d["parity"]["queries"] == 5 and d["parity"]["max_abs_score_diff"] == 0.0
    assert d["self_parity"]["ids_identical"] == d["self_parity"]["queries"]
    assert 0.0 <= d["recall_at_k"] <= 1.0 and d["recall_queries"] == 6
    assert d["maxsim"]["frac_of_hbm_peak"] > 0 and "approx16" in d["roofline_all"]


def test_reference_arm_contract():
    d = _run(["--impl", "reference"])
    assert d["impl"] == "reference" and d["cpu_baseline"]["kind"] == "port" and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] and d["cpu_baseline"]["cores"] >= 1


def _dump(tmp_path, name, extra):
    d = _run(extra + ["--dump-outputs", str(tmp_path / name)])
    return d, {n: np.load(tmp_path / name / f"{n}.npy") for n in ("passage_ids", "scores", "counts")}


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    d3, a = _dump(tmp_path, "a", [])
    _, b = _dump(tmp_path, "b", [])
    _, ref = _dump(tmp_path, "ref", ["--impl", "reference"])
    d2, two = _dump(tmp_path, "two", ["--steps", "2"])
    assert sorted(os.listdir(tmp_path / "a")) == ["counts.npy", "passage_ids.npy", "scores.npy"]
    assert (a["passage_ids"].dtype, a["scores"].dtype, a["counts"].dtype) == (np.float64, np.float32, np.float64)
    assert a["passage_ids"].shape == a["scores"].shape == (4, 5) and a["counts"].shape == (4,)
    n = a["counts"].astype(int)
    assert (n > 0).all() and all((a["passage_ids"][i, n[i]:] == -1).all() for i in range(4))
    # the same arguments give the same inputs and outputs; the stand-in is the oracle, so the reference arm's last
    # step (the same queries) returns the same arrays
    for x in (b, ref):
        assert all(np.array_equal(a[k], x[k]) for k in a)
    # --steps sets the number of timed steps, and so which batch the last one searched
    assert d3["steps"] == 3 and d2["steps"] == 2 and d2["gpu_launches"] * 3 == d3["gpu_launches"] * 2
    assert not np.array_equal(a["passage_ids"], two["passage_ids"])


def test_dump_outputs_samples_rows_above_the_size_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(sys, "dont_write_bytecode", sys.dont_write_bytecode)   # bench.py sets it on import
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 64 * 1024)
    B, k = 1000, 10
    ids = np.arange(B * k, dtype=np.int64).reshape(B, k)
    counts = np.full(B, k, np.int64)
    counts[::7] = 3
    bench.dump_outputs(str(tmp_path / "x"), ids, ids.astype(np.float32) / 2, counts)
    bench.dump_outputs(str(tmp_path / "y"), ids, ids.astype(np.float32) / 2, counts)
    got = {n: np.load(tmp_path / "x" / f"{n}.npy") for n in ("passage_ids", "scores", "counts", "rows")}
    assert sum(os.path.getsize(tmp_path / "x" / f) for f in os.listdir(tmp_path / "x")) <= 64 * 1024 + 4 * 128
    rows = got["rows"].astype(np.int64)
    assert 0 < len(rows) < B and (np.diff(rows) > 0).all()
    assert np.array_equal(got["counts"], counts[rows])
    want = np.where(np.arange(k)[None, :] < counts[rows, None], ids[rows], -1)
    assert np.array_equal(got["passage_ids"], want) and np.array_equal(got["scores"], np.where(want < 0, 0, want / 2))
    assert all(np.array_equal(got[n], np.load(tmp_path / "y" / f"{n}.npy")) for n in got)
