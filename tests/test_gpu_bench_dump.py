"""bench.py --dump-outputs: the arrays written after the timed steps are what the last timed build computed, checked
against the oracle on the same seeded text (a text larger than the row sample, so the sampled path is the one run)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle as O

pytestmark = pytest.mark.gpu


def test_dump_outputs_match_the_oracle(cuda, tmp_path):
    import bench
    size, steps = 1_000_000, 2
    out_dir = tmp_path / "outputs"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--size", str(size), "--no-queries", "--no-c3", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["config"]["text_bytes"] == size

    got = {f[:-4]: np.load(out_dir / f) for f in os.listdir(out_dir)}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20

    kind, seed, _, _ = bench.WORKLOADS["c2"]
    t = O.gen_text(kind, seed, size).tobytes() + b"$"
    n = len(t)
    sa = O.build_suffix_array(t)
    bwt = O.bwt_transform(t, sa)
    rows = got["rows"].astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS < n and bool((np.diff(rows) > 0).all()) and rows[-1] < n
    assert np.array_equal(got["sa"], sa[rows]) and np.array_equal(got["sa_via_samples"], sa[rows])
    assert np.array_equal(got["bwt"], bwt[rows])
    want_occ = np.empty(len(rows), dtype=np.int64)
    for c in np.unique(bwt):
        at = bwt[rows] == c
        want_occ[at] = np.cumsum(bwt == c)[rows[at]] - 1          # occurrences of c before the row
    assert np.array_equal(got["occ"], want_occ)
    _, spine = O.wt_spine(bwt)
    levels = sum(k.startswith("wt_level") for k in got)
    assert levels >= len(spine) and {f"wt_level{l}" for l in range(levels)} <= set(got)
    for l, bits in enumerate(spine):                               # the reference's spine: prefixes of our levels
        below = rows[rows < len(bits)]
        assert np.array_equal(got[f"wt_level{l}"][: len(below)], bits[below])
    assert {chr(int(c)): int(v) for c, v in got["count"]} == O.count_dict(t)
