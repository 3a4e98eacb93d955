"""bench.py --dump-outputs: the proofs of the last timed steps are written as float32 arrays, are valid proofs of the benchmarked
instance, and are identical between two runs with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, BENCH, "--steps", "0"], capture_output=True, text=True, timeout=60)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.gpu
def test_dump_outputs_are_valid_and_repeatable(tmp_path):
    import verify_saved_proof as vsp
    args = ["--log-n", "10", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-verify"]
    runs = []
    for i in range(2):
        d = tmp_path / f"run{i}"
        proof_json = tmp_path / f"proof{i}.json"
        out = subprocess.run([sys.executable, BENCH, *args, "--dump-outputs", str(d), "--save-proof", str(proof_json)], capture_output=True,
                             text=True, timeout=600)
        assert out.returncode == 0, out.stderr
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and len(line["dev_ms_steps"]) == 2
        dumped = {}
        for name in ("proof", "proof_e2e"):
            a = np.load(d / f"{name}.npy")
            assert a.dtype == np.float32 and a.ndim == 1 and len(a) == line["proof_bytes"]
            assert np.all((a >= 0) & (a <= 255) & (a == np.round(a)))
            dumped[name] = a.astype(np.uint8).tobytes()
        assert dumped["proof"] != dumped["proof_e2e"]  # the zk stream moves on between the two timed regions
        blob = json.loads(proof_json.read_text())
        for proof in dumped.values():
            res = vsp.verify_blob(dict(blob, proof_hex=proof.hex()), use_pairing=False)
            assert res["trapdoor"] and res["trapdoor_rejects_wrong_input"]
        runs.append(dumped)
    assert runs[0] == runs[1]
