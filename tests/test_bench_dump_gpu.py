"""bench.py --dump-outputs on the GPU: the dumped arrays are the results of the timed path's last step (every batch of
it, in order), checked against the exact fp64 oracle on the same seeded corpus and queries; --steps sets the timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from helpers import assert_topk_matches
from oracle import dense as dense_oracle
from sentio_b200 import synth

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(built_lib, tmp_path):
    n, d, k, B, inner, steps = 20000, 256, 100, 256, 3, 2
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--n-docs", str(n), "--dim", str(d),
           "--top-k", str(k), "--batch", str(B), "--inner", str(inner), "--steps", str(steps), "--warmup", "1",
           "--no-extras", "--cpu-sample", "0", "--dump-outputs", str(tmp_path)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = out.stdout.splitlines()
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    assert line["steps"] == steps and line["config"]["batches_per_step"] == inner
    ids, sc, cnt = (np.load(tmp_path / f"{name}.npy") for name in ("ids", "scores", "counts"))
    assert ids.dtype == sc.dtype == cnt.dtype == np.float64
    assert ids.shape == sc.shape == (inner * B, k) and cnt.shape == (inner * B,)
    assert not (tmp_path / "query_rows.npy").exists()
    # the bench cycles ring = 1024 // B distinct batches of its 1024 seeded queries; batch j holds queries j*B .. j*B+B-1
    ring = min(8, 1024 // B)
    q = synth.query_vectors(1024, d)
    rows16 = dense_oracle.stored_rows(synth.dense_corpus(n, d))
    for r in range(inner):
        j = ((steps - 1) * inner + r) % ring
        for i in range(0, B, 5):
            row = r * B + i
            wi, ws = dense_oracle.dense_topk(rows16, q[(j * B + i) % 1024], k)
            assert_topk_matches(ids[row].astype(np.int64), sc[row], int(cnt[row]), wi, ws, what=f"batch {r} query {i}")
