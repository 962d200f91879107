"""bench.py contract: the reference arm prints exactly one JSON line with the keys a caller reads, whatever else libraries
write (stdout is reserved for that line); on the GPU, --dump-outputs writes what the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "codewords/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"] == "viterbi_k7_n1024_hard" and d["value"] > 0


def test_arguments_without_a_timed_step_or_a_dump_are_rejected():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                           timeout=120, cwd=ROOT)
        assert r.returncode == 2 and r.stdout == "", (extra, r.stderr[-500:])


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """--dump-outputs: float arrays of at most 64 MB in all, identical for identical inputs whatever the number of steps;
    every step decodes the same frames, so the last step's error counters are the run's totals over the steps"""
    dumps = []
    for steps in (1, 2):
        out = tmp_path / ("steps%d" % steps)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                            "--no-extras", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads(r.stdout)
        assert d["steps"] == steps
        arrays = {f: np.load(out / f) for f in sorted(os.listdir(out))}
        assert sorted(arrays) == ["decoded_bits.npy", "error_counters.npy"]
        assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        dec, cnt = arrays["decoded_bits.npy"], arrays["error_counters.npy"]
        assert dec.shape == (16, 512, 1024) and set(np.unique(dec)) <= {0.0, 1.0}
        assert cnt[0] * steps == d["result"]["bit_errors"] and cnt[1] * steps == d["result"]["frame_errors"]
        assert 0 < cnt[0] < 1e-2 * 16 * 65536 * 1024
        dumps.append(arrays)
    for name in dumps[0]:
        np.testing.assert_array_equal(dumps[0][name], dumps[1][name], err_msg=name)
