"""-m gpu: `bench.py --dump-outputs` writes the headline's results block of the last timed step, and that block equals the
CPU oracle's group table on the same seeded table."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    import bench
    from pinot_b200 import sql
    segments, rows = 2, 1_000_000
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--steps", "2", "--warmup", "1",
                        "--segments", str(segments), "--rows", str(rows), "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(got) == {"group_keys", "agg0_sum_c5", "agg1_count"}
    assert all(a.dtype == np.float64 for a in got.values())
    keys = got["group_keys"][:, 0].astype(np.int64)
    assert np.all(np.diff(keys) > 0), "rows ordered by key"

    _, tables = bench.CpuTable(segments, rows, 0, 4).run(sql.parse(bench.groupby_query_text(0.10)))
    want = {}
    for t in tables:
        for k, (s, c) in t.items():
            cur = want.setdefault(k, [0.0, 0])
            cur[0] += s
            cur[1] += c
    dumped = {int(k): [float(s), int(c)] for k, s, c in zip(keys, got["agg0_sum_c5"], got["agg1_count"])}
    bench.assert_same_table(dumped, want, "dumped block vs CPU oracle")
