"""A/B comparison of two builds of this repository on one GPU.

    python tools/ab_bench.py --old OLD_TREE --new NEW_TREE --out DIR [--rounds 3] [--extra-rounds 1]

OLD_TREE and NEW_TREE are two built checkouts (each with its own marlin_b200/libb2m.so).  The script
  1. records the card (name, power limit, max SM clock) once;
  2. runs `bench.py --steps 10 --warmup 3` (the flagship: 2^20 constraints, BLS12-381, MarlinKZG10) alternately from the old
     and the new tree, --rounds times each, and prints the median ms_per_step of each and the min / max of every run;
  3. runs SonicKZG10 2^20, BN254 2^20 and SonicKZG10 2^22 old / new alternately, --extra-rounds times each;
  4. compares the proofs `bench.py --dump-outputs` wrote for the first flagship run of each tree;
  5. reads the peak size of the device's default memory pool (the pool libb2m allocates from) over one 2^20 set-up + prove in
     a fresh process per tree (`--pool-peak TREE`).
Every bench line is written to DIR/ab_lines.jsonl with the tree and round, the summary to DIR/ab_summary.json.  Nothing is
written into either tree.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))


def pool_peak(tree):
    """One 2^20 MarlinKZG10 set-up + index + two proves from `tree`; the default pool's high-water marks, in bytes."""
    sys.path.insert(0, tree)
    from marlin_b200 import _lib, api, r1cs
    _lib.lib()  # loads libb2m.so and with it libcudart.so.12, which the lookup below then finds
    rt = ctypes.CDLL("libcudart.so.12")
    RESERVED_HIGH, USED_HIGH = 0x6, 0x8  # cudaMemPoolAttrReservedMemHigh, cudaMemPoolAttrUsedMemHigh

    def attr(pool, a):
        v = ctypes.c_uint64(0)
        assert rt.cudaMemPoolGetAttribute(pool, a, ctypes.byref(v)) == 0
        return v.value

    n = 1 << 20
    m = api.Marlin("bls12_381", "marlin_kzg10", device=0)
    pool = ctypes.c_void_p()
    assert rt.cudaDeviceGetDefaultMemPool(ctypes.byref(pool), 0) == 0
    circ = r1cs.dummy_circuit(m.curve_id, 0x1234567890abcdef1234567890abcdef, 0xfedcba0987654321fedcba0987654321, 10, n)
    srs = m.universal_setup(n, n, 3 * n, beta=0x5eed5eed5eed5eed5eed5eed, gamma=7, degree_bounds=(n - 2, 4 * n - 2))
    pk = m.index(srs, circ)
    m.stage(pk, circ)
    after_setup = {"reserved_high": attr(pool, RESERVED_HIGH), "used_high": attr(pool, USED_HIGH)}
    zero = ctypes.c_uint64(0)  # writing 0 resets a high-water mark to the current value
    assert rt.cudaMemPoolSetAttribute(pool, USED_HIGH, ctypes.byref(zero)) == 0
    for _ in range(2):
        m.prove(pk, None, api.ZkRng.test_rng())
    used_prove = attr(pool, USED_HIGH)
    out = {"after_setup": after_setup, "reserved_high_total": attr(pool, RESERVED_HIGH), "used_high_during_prove": used_prove,
           "prove_scratch_above_setup": used_prove - after_setup["used_high"] if used_prove > after_setup["used_high"] else 0}
    pk.close()
    srs.close()
    print(json.dumps(out))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def bench(tree, args, dump=None):
    cmd = [sys.executable, "bench.py", "--no-cpu-baseline"] + args
    if dump:
        cmd += ["--dump-outputs", dump]
    t0 = time.time()
    p = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    if p.returncode != 0 or not lines:
        raise RuntimeError(f"bench failed in {tree}: {p.returncode}\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}")
    line = json.loads(lines[-1])
    line["_wall_s"] = time.time() - t0
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old")
    ap.add_argument("--new")
    ap.add_argument("--out")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--extra-rounds", type=int, default=1)
    ap.add_argument("--pool-peak", metavar="TREE", help="(internal) print the pool high-water marks of one 2^20 prove from TREE")
    a = ap.parse_args()
    if a.pool_peak:
        pool_peak(os.path.abspath(a.pool_peak))
        return
    old, new = os.path.abspath(a.old), os.path.abspath(a.new)
    os.makedirs(a.out, exist_ok=True)
    trees = (("old", old), ("new", new))
    gpu = card()
    print("card:", gpu, flush=True)
    rec = open(os.path.join(a.out, "ab_lines.jsonl"), "w")

    def run(tag, tree, rnd, cfg, args, dump=None):
        ln = bench(tree, args, dump)
        ln.update({"_tree": tag, "_round": rnd, "_config": cfg, "_card": gpu})
        rec.write(json.dumps(ln) + "\n")
        rec.flush()
        print(f"{cfg:>16} {tag} r{rnd}: {ln['ms_per_step']:.2f} ms  sha {ln['proof_sha256'][:8]}  pinned {ln['proof_matches_pinned_1gpu_hash']}  "
              f"verified {ln['proof_verified']}  clocks {json.dumps(ln['clocks'])}", flush=True)
        return ln

    flag = {"old": [], "new": []}
    for r in range(a.rounds):
        for tag, tree in trees:
            dump = os.path.join(os.path.abspath(a.out), "dump_" + tag) if r == 0 else None
            flag[tag].append(run(tag, tree, r, "flagship", ["--steps", "10", "--warmup", "3"], dump))
    extra = {}
    for cfg, args in (("sonic_2p20", ["--pc", "sonic_kzg10"]), ("bn254_2p20", ["--curve", "bn254"]),
                      ("sonic_2p22", ["--pc", "sonic_kzg10", "--log-n", "22"])):
        for r in range(a.extra_rounds):
            for tag, tree in trees:
                extra.setdefault(cfg, {}).setdefault(tag, []).append(run(tag, tree, r, cfg, ["--steps", "10", "--warmup", "3"] + args))
    same_dump = all(open(os.path.join(a.out, "dump_old", f), "rb").read() == open(os.path.join(a.out, "dump_new", f), "rb").read()
                    for f in ("proof.npy", "proof_e2e.npy"))
    pool = {}
    for tag, tree in trees:
        p = subprocess.run([sys.executable, os.path.join(HERE, "ab_bench.py"), "--pool-peak", tree], cwd=tree, capture_output=True, text=True)
        pool[tag] = json.loads(p.stdout.strip().splitlines()[-1]) if p.returncode == 0 else {"error": p.stderr[-2000:]}
    ms = {t: [ln["ms_per_step"] for ln in flag[t]] for t in flag}
    summary = {
        "card": gpu,
        "flagship_ms": ms,
        "flagship_median_ms": {t: statistics.median(v) for t, v in ms.items()},
        "median_gain_ms": statistics.median(ms["old"]) - statistics.median(ms["new"]),
        "every_new_faster_than_every_old": max(ms["new"]) < min(ms["old"]),
        "flagship_clocks": {t: [ln["clocks"] for ln in flag[t]] for t in flag},
        "flagship_bucket_spans_ms_per_step": {t: [{k: v["ms"] / ln["steps"] for k, v in ln["kernels"].items()} for ln in flag[t]][0] for t in flag},
        "hashes": sorted({ln["proof_sha256"] for t in flag for ln in flag[t]}),
        "pinned_and_verified": all(ln["proof_matches_pinned_1gpu_hash"] and ln["proof_verified"] for t in flag for ln in flag[t]),
        "dump_outputs_identical": same_dump,
        "extra": {cfg: {t: {"ms": [ln["ms_per_step"] for ln in v], "sha": sorted({ln["proof_sha256"] for ln in v}),
                            "pinned": [ln["proof_matches_pinned_1gpu_hash"] for ln in v], "verified": [ln["proof_verified"] for ln in v]}
                        for t, v in d.items()} for cfg, d in extra.items()},
        "pool_peak_bytes": pool,
    }
    with open(os.path.join(a.out, "ab_summary.json"), "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
