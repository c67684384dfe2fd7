"""bench.py's contract: the reference arm on CPU exits 0 and prints ONE JSON line with the keys a results reader
needs; on a GPU, --dump-outputs writes what the last timed step returned."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env):
    env = dict(os.environ, AUR_BENCH_ROWS="16000", **extra_env)      # (the real arm scans the full 1M rows per step)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                          capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)


def test_reference_arm_prints_one_json_line():
    p = _run({})
    assert p.returncode == 0, p.stderr[-500:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["metric"].startswith("RAG queries/sec")
    assert d["config"]["rows"] == 16_000 and d["config"]["dim"] == 768 and d["config"]["k"] == 32 and d["config"]["nq"] == 256
    assert "no extrapolation" in d["cpu_baseline"]["sample"] and d["cpu_baseline"]["threads"] >= 1
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_nonzero_ranks_exit_quietly():
    p = _run({"RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_is_refused_where_it_is_not_implemented(tmp_path):
    for argv in (["--impl", "reference"], ["--config", "cfg3"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv, "--dump-outputs", str(tmp_path / "out")],
                           capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert p.returncode == 2 and "--dump-outputs" in p.stderr and not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    out = tmp_path / "out"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--no-parity",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == 2
    ids, sc, emb = (np.load(out / f"{n}.npy") for n in ("topk_ids", "topk_scores", "encoder_embeddings"))
    assert ids.dtype == np.float64 and ids.shape == (256, 32) and sc.dtype == np.float32 and sc.shape == (256, 32)
    assert np.all(ids == np.rint(ids)) and ids.min() >= 0 and ids.max() < 1_000_000
    assert all(len(set(r)) == 32 for r in ids) and np.all(np.diff(sc, axis=1) <= 0)      # distinct rows, best first
    assert emb.dtype == np.float32 and emb.shape == (192, 768) and np.all(np.isfinite(emb))
    assert sorted(os.listdir(out)) == ["encoder_embeddings.npy", "topk_ids.npy", "topk_scores.npy"]
