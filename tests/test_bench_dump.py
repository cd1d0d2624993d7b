"""GPU: bench.py --dump-outputs writes the same arrays from run to run and for any --steps (every step computes a fresh
population of connections from the same seeded input), within its size limit, and what it writes is what the oracle
computes for the sampled connections."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from inference_gateway_b200 import _abi as A
from inference_gateway_b200 import synth
from oracle import orc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_STREAMS = 512


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--streams", str(N_STREAMS), "--steps", str(steps), "--warmup", "3",
           "--segments", "0", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    a, b = run_bench(tmp_path / "a", 2), run_bench(tmp_path / "b", 5)
    assert sorted(a) == sorted(b) == ["connections", "content_bytes", "frame_bytes", "frame_len", "records", "sample",
                                      "tool_call_bytes", "tool_calls"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= 64_000_000
    bodies = [s for s, _, _ in synth.make_config("C4", n_streams=N_STREAMS)[0]]
    assert len(a["connections"]) == len(a["sample"]) == N_STREAMS
    conns = a["sample"][:, 0].astype(int)
    assert sorted(conns) == list(range(N_STREAMS))
    frames = a["frame_bytes"].astype(np.uint8).tobytes()
    flen = a["frame_len"].astype(int)
    pos = np.concatenate([[0], np.cumsum(flen)])
    f0 = np.concatenate([[0], np.cumsum(a["sample"][:, 1].astype(int))])
    recs = a["records"]
    for i, c in enumerate(conns):
        v = orc.reframe(bodies[c])
        exp = [l.out for l in v.lines if l.kind == orc.L_EMITTED]
        got = [frames[pos[k]:pos[k + 1]] for k in range(f0[i], f0[i + 1])]
        assert got == exp, f"connection {c}"
        row = a["connections"][np.searchsorted(a["connections"][:, 0], c)]
        assert row[3] == len(exp) and row[4] == sum(map(len, exp))
        assert bool(int(row[2]) & A.SEG_TERMINATED) == v.terminated
        mine = recs[recs[:, 0] == c]
        assert len(mine) == row[5] == a["sample"][i, 2]
    ok = recs[:, 2].astype(int) & A.F_JSON_OK != 0
    assert ok.any() and recs[ok, 8].sum() == len(a["content_bytes"])
    assert len(a["tool_calls"]) and a["tool_calls"][:, 5:].sum() == len(a["tool_call_bytes"])
