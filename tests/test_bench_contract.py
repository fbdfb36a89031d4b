"""bench.py's output: the keys of its one JSON result line (reference arm, on the CPU) and the arrays --dump-outputs
writes (CUDA arm, on the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--ref-sample-gb", "0.03"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("GB/s SHA-256-digested on 100 GB")
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and "workload" in d["config"]
    assert d["native_so_loaded"] is False          # VERDICT r1 item 11: the reference arm must not map the product library


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1", "--ref-sample-gb", "0.03"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_are_the_digests_of_the_timed_step(oracle, tmp_path):
    """--dump-outputs writes the chunk digests and the root the timed steps computed, as float32 arrays of byte values;
    they are the tree digest of the seeded blob, so two runs or two builds can be compared array for array."""
    size, tp = 100_000_000, (8 << 20, 16 << 10, 8)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--size", str(size),
                          "--no-e2e", "--no-cpu", "--no-compat", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    chunks, root = np.load(tmp_path / "chunk_digests.npy"), np.load(tmp_path / "root.npy")
    assert chunks.dtype == np.float32 and chunks.shape == (12, 32) and root.dtype == np.float32 and root.shape == (32,)
    want_chunks, _, want_root = oracle.tree_digest(oracle.gen(0, size, 0x6D6F64656C78), *tp)
    assert chunks.astype(np.uint8).tobytes() == b"".join(want_chunks)
    assert root.astype(np.uint8).tobytes() == want_root
    assert d["root"] == oracle.digest_string(want_root) and d["steps"] == 2
