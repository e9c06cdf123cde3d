"""bench.py contract on CPU: the reference arm prints ONE JSON line with the keys the driver reads (metric, unit,
value, impl, cpu_baseline, e2e with zero copies), and the files README/DESIGN cite under profiles/ exist."""
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "end-to-end PPO env-steps/sec" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_dump_outputs_sample_below_cap(tmp_path, monkeypatch):
    """--dump-outputs with a rollout buffer larger than the cap: a seeded sample of env columns, float32 / float64 files only,
    within the cap, the same columns every time."""
    import importlib.util

    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from dril_b200 import _lib as L
    T, N = 8, 1000

    class Buf:
        n_envs = N

        def download(self, f):
            shape = {"obs": (T, N, 4), "actions": (T, N, 1), "last_values": (N,)}.get(f, (T, N))
            dt = {"flags": np.uint8, "episode_l": np.int32, "actions": np.int32}.get(f, np.float32)
            return np.arange(np.prod(shape)).reshape(shape).astype(dt)

    class Agent:
        class device:
            get_params = staticmethod(lambda: np.ones(100, np.float32))

    monkeypatch.setattr(bench, "DUMP_BYTES", 200_000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), Agent, Buf(), L.IterStats())
    names = sorted(os.listdir(tmp_path / "a"))
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 200_000
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert 0 < idx.size < N and (np.diff(idx) > 0).all()
    np.testing.assert_array_equal(idx, np.load(tmp_path / "b" / "env_index.npy"))
    for n in names:
        assert np.load(tmp_path / "a" / n).dtype in (np.float32, np.float64), n
    obs = np.load(tmp_path / "a" / "buf_obs.npy")
    np.testing.assert_array_equal(obs, Buf().download("obs")[:, idx.astype(int)])
    assert "stat_rollout_ms.npy" not in names and "stat_loss.npy" in names


def test_cited_profile_files_exist():
    cited = set()
    for doc in ("README.md", "DESIGN.md", os.path.join("profiles", "README.md")):
        text = open(os.path.join(ROOT, doc)).read()
        cited |= set(re.findall(r"profiles/(r01_[A-Za-z0-9_]+\.(?:json|csv|txt))", text))
        if doc.startswith("profiles"):
            cited |= set(re.findall(r"`(r01_[A-Za-z0-9_]+\.(?:json|csv|txt))`", text))
    assert cited, "no profile files cited"
    missing = sorted(f for f in cited if not os.path.exists(os.path.join(ROOT, "profiles", f)))
    assert not missing, missing
