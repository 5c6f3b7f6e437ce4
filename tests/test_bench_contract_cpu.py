"""bench.py contract, CPU side: the reference arm runs without a GPU and prints ONE JSON line with the keys the driver
reads (impl / metric / unit / value / steps / warmup / e2e / cpu_baseline / config)."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT


def _run(*extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--n-docs", "6000", "--dim", "64",
           "--steps", "2", "--warmup", "1", *extra]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    # stdout carries the result line and NOTHING else (library banners such as NCCL's are routed to stderr)
    lines = out.stdout.splitlines()
    assert len(lines) == 1 and lines[0].startswith("{"), out.stdout
    return json.loads(lines[0])


def test_reference_arm_prints_one_contract_line():
    d = _run()
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("retrieval queries/sec") and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1 and d["data"] == "synthetic"
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_reference_arm_hybrid_workload():
    d = _run("--workload", "hybrid")
    assert "hybrid dense+BM25 rrf" in d["config"]["workload"] and "BM25" in d["cpu_baseline"]["sample"]


_DUMP = """
import importlib.util, os, sys
import numpy as np
import torch

spec = importlib.util.spec_from_file_location("bench", sys.argv[1])
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)
bench.DUMP_LIMIT_BYTES = int(sys.argv[3])
g = torch.Generator().manual_seed(0)
ids = torch.randint(0, 1 << 40, (6, 50, 10), dtype=torch.int64, generator=g)
sc = torch.rand((6, 50, 10), dtype=torch.float64, generator=g)
cnt = torch.randint(0, 11, (6, 50), dtype=torch.int32, generator=g)
bench.dump_outputs(sys.argv[2], "dense", [ids, sc, cnt])
np.savez(os.path.join(sys.argv[2], "want.npz"), ids=ids.numpy(), sc=sc.numpy(), cnt=cnt.numpy())
"""


def _dump(path, limit):
    out = subprocess.run([sys.executable, "-c", _DUMP, os.path.join(ROOT, "bench.py"), str(path), str(limit)],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    want = np.load(path / "want.npz")
    got = {n: np.load(path / f"{n}.npy") for n in ("ids", "scores", "counts")}
    assert all(a.dtype == np.float64 for a in got.values())
    rows = np.load(path / "query_rows.npy").astype(np.int64) if (path / "query_rows.npy").exists() else np.arange(300)
    assert np.array_equal(got["ids"], want["ids"].reshape(300, 10)[rows])        # int64 ids survive float64 exactly
    assert np.array_equal(got["scores"], want["sc"].reshape(300, 10)[rows])
    assert np.array_equal(got["counts"], want["cnt"].reshape(300)[rows])
    return rows, sum((path / f"{n}.npy").stat().st_size for n in ("ids", "scores", "counts", "query_rows")
                     if (path / f"{n}.npy").exists())


def test_dump_outputs_writes_the_last_step_rows_in_order_under_the_size_cap(tmp_path):
    """bench.py --dump-outputs: every batch of the step, in order, as float64; above the cap a fixed seeded row sample."""
    rows, _ = _dump(tmp_path / "all", 64 << 20)
    assert np.array_equal(rows, np.arange(300)) and not (tmp_path / "all" / "query_rows.npy").exists()
    limit = (1 << 20) + 20_000
    a, size = _dump(tmp_path / "a", limit)
    b, _ = _dump(tmp_path / "b", limit)
    assert 0 < len(a) < 300 and size <= limit and np.array_equal(a, b)
