"""`bench.py --dump-outputs DIR`: the arrays it writes are exactly the proof of the last timed step (float64, each u64 as
its [low, high] 32-bit halves), so that two builds can be compared output for output.  Each arm is checked against the
oracle prover on the same seeded workload at a small height."""
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H
import oracle_binding as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _u64(path):
    a = np.load(path)
    assert a.dtype == np.float64 and a.shape[-1] == 2
    assert np.all(a >= 0) and np.all(a < 2.0 ** 32) and np.all(a == np.floor(a))
    return a[..., 0].astype(np.uint64) | (a[..., 1].astype(np.uint64) << np.uint64(32))


def _bench_dump(tmp_path, *args):
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-1500:]
    assert sorted(os.listdir(out)) == ["commitments.npy", "fields.npy", "log_trace_heights.npy"]
    heights = np.load(out / "log_trace_heights.npy")
    assert heights.dtype == np.float64
    return bytes(heights.astype(np.uint8)), _u64(out / "fields.npy"), _u64(out / "commitments.npy")


def _assert_is_the_oracle_proof(dumped, log_height):
    params = H.W.miden_pcs_params()
    wl = H.W.Workload([log_height] * 3)
    ch = H.W.initial_challenger(params, H.oracle_observe)
    h, heights, fields, comms = H.oracle_prove(params, wl, ch)
    ob.lib().orc_prove_free(h)
    assert dumped[0] == heights
    assert np.array_equal(dumped[1], fields) and np.array_equal(dumped[2], comms)


def test_reference_arm_dumps_its_last_proof(tmp_path):
    dumped = _bench_dump(tmp_path, "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1", "--ref-log-height", "10")
    _assert_is_the_oracle_proof(dumped, 10)


@pytest.mark.gpu
def test_cuda_arm_dumps_its_last_proof(tmp_path):
    dumped = _bench_dump(tmp_path, "--gpus", "1", "--steps", "2", "--warmup", "1", "--log-height", "12", "--no-cpu-baseline")
    _assert_is_the_oracle_proof(dumped, 12)
