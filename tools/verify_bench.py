#!/usr/bin/env python3
"""Batch-verification throughput of `Marlin.batch_verify` on one GPU; prints one JSON line.

For each configuration (curve, PC scheme, 2^log_n-constraint DummyCircuit) it proves `--distinct` proofs, tiles them to batches
of N proofs and times `batch_verify` (host clock around the call, which returns after the device has finished), after one
warm-up call per N.  Per-stage times are the verifier's own (CUDA events for the device stages, host clock for the
transcripts) from the last timed call.  The card name and power limit are read with a read-only nvidia-smi query."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from marlin_b200 import api, fields, r1cs as gr1cs  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception:  # noqa: BLE001 -- the numbers stay valid without the label
        return "unknown", "unknown"


def run_config(ctx, curve, pc, log_n, ns, distinct, reps):
    n = 1 << log_n
    cid = fields.CURVE_IDS[curve]
    r = fields.FR_MODULUS[cid]
    m = api.Marlin(curve, pc, ctx=ctx)
    srs = m.universal_setup(n, n, 3 * n, beta=0x5eed5eed5eed5eed5eed, gamma=7, degree_bounds=(n - 2, 4 * n - 2))
    a, b = 0x1234567 % r, 0x7654321 % r
    circ = gr1cs.dummy_circuit(cid, a, b, 10, n)
    pk = m.index(srs, circ)
    vk = m.verifier_key(pk)
    zk = api.ZkRng(bytes(range(32)), 12)
    proofs = [m.prove(pk, circ, zk) for _ in range(distinct)]
    pub = [a * b % r]
    out = []
    for N in ns:
        items = [(pub, proofs[i % distinct]) for i in range(N)]
        rng = api.ZkRng(bytes([9] * 32), 12)
        assert all(m.batch_verify(vk, items, rng))
        times = []
        for _ in range(reps):
            t0 = time.perf_counter()
            ok = m.batch_verify(vk, items, rng)
            times.append(time.perf_counter() - t0)
            assert all(ok)
        best = min(times)
        out.append({"curve": curve, "pc": pc, "log_n": log_n, "n_proofs": N, "distinct_proofs": distinct, "best_s": round(best, 6),
                    "median_s": round(sorted(times)[len(times) // 2], 6), "proofs_per_s": round(N / best, 1), "stages_ms": vk.timings()})
    vk.close()
    pk.close()
    srs.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log-n", type=int, nargs="+", default=[10, 16])
    ap.add_argument("--n", type=int, nargs="+", default=[1, 64, 1024, 4096])
    ap.add_argument("--distinct", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="bls12_381:marlin_kzg10,bls12_381:sonic_kzg10,bn254:marlin_kzg10")
    args = ap.parse_args()
    name, power = card()
    ctx = api.Context(0)
    results = []
    for cfg in args.configs.split(","):
        curve, pc = cfg.split(":")
        for log_n in args.log_n:
            results += run_config(ctx, curve, pc, log_n, args.n, args.distinct, args.reps)
    print(json.dumps({"tool": "verify_bench", "gpu": name, "power_limit": power, "timing": "host clock around batch_verify (device-synchronous)",
                      "results": results}))


if __name__ == "__main__":
    main()
