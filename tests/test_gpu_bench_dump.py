"""bench.py --dump-outputs: the arrays written are what the last timed step returned to its caller.  The
step is recomputed here from the bench's own seeds: with --warmup 1 --steps 2 the last timed step is the
third step run, so a dump from any other step (or a run that ignored --steps) does not match."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_last_timed_step(ctx, pkg, tmp_path):
    B = 16
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--batch", str(B), "--no-msm", "--no-latency", "--no-config4", "--no-n512",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2 and line["warmup"] == 1

    files = sorted(tmp_path.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    got = {f.stem: np.load(f) for f in files}
    assert set(got) == {"sample_index", "post_trackers", "proofs", "generate_status", "valid", "validate_status"}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert (got["generate_status"] == 0).all() and (got["valid"] == 1).all() and (got["validate_status"] == 0).all()

    sys.path.insert(0, ROOT)
    import bench

    crs = ctx.generate_crs(bench.ELL, pkg.Rand(0))
    sets = bench.make_trackers(ctx, pkg, bench.ELL, [1000 + i for i in range(8)])
    pre = b"".join(sets[i % len(sets)] for i in range(B))
    post, proofs, status = ctx.whisk_generate_shuffle_proof_batch(crs, pre, [pkg.Rand((2 << 20) | i) for i in range(B)])
    assert status == [0] * B
    idx = got["sample_index"].astype(np.int64)
    assert (idx == np.arange(B)).all()
    assert (got["post_trackers"] == np.frombuffer(post, np.uint8).reshape(B, -1)).all()
    assert (got["proofs"] == np.frombuffer(proofs, np.uint8).reshape(B, -1)).all()
    crs.close()
