"""bench.py --dump-outputs: the arrays the last timed step returned land in DIR as float64 .npy files, and they are the CPU
chain's answer on the benchmark's own seeded workload (rebuilt here with the same arguments)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCH, BEAMS, MAP_SCANS, PAIRS, STEPS = 16, 16, 6, 2, 3    # bench's single-thread CPU arm takes 16 scans


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    args = ["--batch", str(BATCH), "--beams", str(BEAMS), "--map-scans", str(MAP_SCANS), "--pairs", str(PAIRS),
            "--steps", str(STEPS), "--warmup", "1", "--cpu-sample", str(BATCH), "--no-extras", "--dump-outputs", str(tmp_path)]
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-4000:]
    line = json.loads([s for s in out.stdout.splitlines() if s.startswith("{")][-1])
    assert line["steps"] == STEPS
    got = {n: np.load(tmp_path / f"{n}.npy") for n in ("states", "scan_results", "solve_summary", "constraints")}
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["states"].shape == (BATCH, 16) and got["scan_results"].shape == (BATCH, 25)
    assert got["solve_summary"].shape == (BATCH, 7) and got["constraints"].shape == (PAIRS, 15)

    import bench
    w = bench.build_workload(argparse.Namespace(map_scans=MAP_SCANS, batch=BATCH, beams=BEAMS), 0)
    _, want, _, ok, iters = bench.cpu_chain(w, list(range(BATCH)), 1)
    dt, dr = bench.pose_errors(got["states"], want)
    assert dt.max() < 1e-9 and dr.max() < 1e-6, (dt, dr)
    assert np.abs(got["states"][:, 7:] - want[:, 7:]).max() < 1e-9
    assert all(ok == 1) and got["scan_results"][:, 15].tolist() == [1.0] * BATCH                # dl_scan_result.ok
    assert got["solve_summary"][:, 2].tolist() == iters.astype(np.float64).tolist()            # num_iterations
    # the exchange table: rank 0 owns submap 0; node k searches scan (17 k) mod BATCH
    assert got["constraints"][:, :2].tolist() == [[0.0, float(17 * k % BATCH)] for k in range(PAIRS)]
