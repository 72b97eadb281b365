"""bench.py --dump-outputs: the last timed step's seal and roots land as float64 .npy files, --steps is the number of timed steps,
and the same arguments give the same outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from zktls_b200 import circuit, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    dumped = {n: np.load(os.path.join(out_dir, n + ".npy")) for n in ("seal", "roots")}
    for a in dumped.values():
        assert a.dtype == np.float64 and a.size and (a == np.floor(a)).all() and (a >= 0).all() and (a < 2**32).all()
    return line, dumped


def test_reference_arm_dumps_the_oracle_seal(oracle, tmp_path):
    po2 = 10
    line, got = run_bench(tmp_path, "--impl", "reference", "--po2", str(po2), "--steps", "2", "--warmup", "0")
    assert line["steps"] == 2 and line["steps_capped_by"] is None
    blob = circuit.syn_circuit(**circuit.SYN280).blob()
    io, code, data, accum = synth.trace_a(circuit.SYN280, po2, 0xB200)          # the reference arm's trace
    pr = oracle.Prover(blob)
    pr.begin(po2, io, code, data)
    assert np.array_equal(got["seal"], pr.finish(accum).astype(np.float64))
    assert np.array_equal(got["roots"], pr.roots().astype(np.float64))


@pytest.mark.gpu
def test_device_arm_dumps_the_same_outputs_every_run(tmp_path):
    args = ("--po2", "12", "--steps", "4", "--warmup", "1", "--no-cpu-baseline", "--session-segments", "0")
    line_a, a = run_bench(tmp_path / "a", *args)
    line_b, b = run_bench(tmp_path / "b", *args)
    assert line_a["steps"] == line_b["steps"] == 4
    assert a["seal"].size == line_a["seal_words"] and a["roots"].shape[1] == 8
    assert np.array_equal(a["seal"], b["seal"]) and np.array_equal(a["roots"], b["roots"])
