"""bench.py --dump-outputs on the GPU: the timed steps are exactly --steps iterations, and two runs with the same arguments
write the same arrays (float32 / float64 only, 64 MB at most), so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--repeats", "2",
                          "--no-extra", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_dump_outputs_repeatable(tmp_path):
    runs = [tmp_path / "a", tmp_path / "b", tmp_path / "c"]
    lines = [_bench(runs[0], 4), _bench(runs[1], 4), _bench(runs[2], 3)]
    assert [len(l["block_ms"]) for l in lines] == [2, 2, 1]              # 4 steps in 2 blocks; 3 steps in 1 block
    names = sorted(os.listdir(runs[0]))
    assert names == sorted(os.listdir(runs[1])) == sorted(os.listdir(runs[2]))
    assert {"params.npy", "buf_obs.npy", "buf_advantages.npy", "stat_loss.npy"} <= set(names)
    assert sum(os.path.getsize(runs[0] / n) for n in names) <= 64 * 10 ** 6
    for n in names:
        a, b = np.load(runs[0] / n), np.load(runs[1] / n)
        assert a.dtype in (np.float32, np.float64), n
        np.testing.assert_array_equal(a, b, err_msg=n)
    # one timed step fewer: the last step starts from other parameters
    assert not np.array_equal(np.load(runs[0] / "params.npy"), np.load(runs[2] / "params.npy"))
