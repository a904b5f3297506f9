"""bench.py's reference arm (`--impl reference`) runs on the host alone, so its JSON contract is checked in the CPU tier:
the keys the driver reads, `impl`, a `cpu_baseline` describing the run, an `e2e` that repeats the line's value with no copies."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                        "--batch", "4", "--unique", "2", "--residues", "200000", "--level", "3"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "decoded_ascii_GBps" and line["unit"] == "GB/s"
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["value"] > 0
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    e = line["e2e"]
    assert e["value"] == line["value"] and e["unit"] == line["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.gpu
def test_dumped_outputs_are_the_same_from_run_to_run(tmp_path):
    """--dump-outputs writes what the last timed step decoded; runs with the same workload and a different number of steps
    write the same arrays, and those arrays are the workload's decoded records."""
    import numpy as np
    import _cases as K
    import _oracle as O
    small = ["--warmup", "1", "--batch", "4", "--unique", "2", "--residues", "200000", "--level", "3", "--no-configs"]
    dumps = []
    for steps in (2, 3):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--dump-outputs", str(out)] + small,
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-4000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({p.stem: np.load(p) for p in out.glob("*.npy")})
    a, b = dumps
    assert sorted(a) == ["comments", "ids", "lengths", "n_records", "sequence_sample"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert all(np.array_equal(a[k], b[k]) for k in a)
    # the batch cycles the archives of seeds 1000 and 1001: one record of 200 000 residues each
    want = [O.decode(K.genome(s, 200_000, level=3, mask=True, records=1)) for s in (1000, 1001)]
    assert a["n_records"].tolist() == [1.0] * 4 and a["lengths"].tolist() == [200_000.0] * 4
    assert bytes(a["ids"].astype(np.uint8)) == b"".join(w.id(0) + b"\0" for w in want * 2)
    assert bytes(a["comments"].astype(np.uint8)) == b"".join(w.comment(0) + b"\0" for w in want * 2)
    assert bytes(a["sequence_sample"].astype(np.uint8)) == b"".join(w.sequence for w in want * 2)     # small archives: whole


def test_other_ranks_of_the_reference_arm_do_no_work():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29999")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1",
                        "--batch", "2", "--unique", "1", "--residues", "100000", "--level", "3"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == ""
