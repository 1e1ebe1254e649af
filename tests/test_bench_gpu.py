"""bench.py --dump-outputs on the GPU: the files hold what the last timed step of the headline workload returned."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(rdf, oracle, tmp_path):
    bench = importlib.import_module("bench")
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--skip-e2e",
                        "--skip-cpu", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and line["check"]["count"] == bench.ROWS
    assert np.load(out / "sum.npy").tolist() == [line["check"]["sum"]]
    assert np.load(out / "count.npy").tolist() == [float(line["check"]["count"])]
    c = np.load(out / "c.npy")
    rows = bench.dump_rows(bench.ROWS)
    assert c.dtype == np.float64 and c.shape == rows.shape
    # a and b come from the counter-based generator: the oracle regenerates any row and adds them
    pick = np.linspace(0, rows.size - 1, 256).astype(np.int64)

    def column(col_id):
        vals = [oracle.generate(oracle.F64, 0, -1e3, 1e3, bench.SEED, col_id, int(rows[k]), 1).values[0] for k in pick]
        return oracle.OracleArray(oracle.F64, np.array(vals), None, 0)

    st, want = oracle.col_binary(oracle.ADD, oracle.F64, [column(0)], [column(1)])
    assert st == oracle.OK
    assert np.array_equal(c[pick].view(np.uint64), want[0].values.view(np.uint64))
