#!/usr/bin/env python3
"""bench.py -- Marlin prover throughput on B200 (BASELINE.json metric: prover constraints/sec, BLS12-381).

A "step" is one `Marlin::prove` (reference src/lib.rs:151-311) of the reference bench's DummyCircuit
(benches/bench.rs:25-67) scaled to 2^log_n constraints; SRS generation and `index` are outside the
timed region exactly as in benches/bench.rs:79-101.

  value : constraints / second with the instance (x, w) already resident in HBM (b2m_index_stage)
  e2e   : the same through the public API with HOST buffers -- host->device copy of the instance and
          device->host read of the proof inside the timed region
  roofline     : the dominant kernel (msm_accumulate_kernel) -- algorithmic bytes (128 B per
                 (base, scalar) pair, SURVEY.md section 8d) / CUDA-event kernel time / measured HBM peak
  cpu_baseline : the oracle's C++ restatement of the reference prover (oracle/cport/prover.cpp) timed on this
                 box's host cores (rank 0, N = 1) on a bounded sample: full proves of a 2^16-constraint
                 instance of the same circuit family (~10-30 s of CPU work)
  --impl reference : the same CPU prover on the SAME 2^log_n configuration as the GPU arm (see run_reference)

N > 1 (torchrun, one rank per GPU): every rank runs the prover, each MSM is sharded by base/scalar
chunk and the partial sums are exchanged with one NCCL all-gather per MSM (DESIGN.md "Multi-GPU");
total work is fixed => "scaling": "strong".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--log-n", type=int, default=20, help="log2 of the number of constraints (BASELINE config 2: 20)")
    ap.add_argument("--pc", default="marlin_kzg10", choices=["marlin_kzg10", "sonic_kzg10"])
    ap.add_argument("--curve", default="bls12_381", choices=["bls12_381", "bn254"])
    ap.add_argument("--cpu-log-n", type=int, default=16, help="instance size of the bounded cpu_baseline sample of the GPU arm's line")
    ap.add_argument("--ref-log-n", type=int, default=0, help="--impl reference: instance size (0 = the same 2^log_n as the GPU arm)")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="--impl reference: stop starting new proves once set-up + proves "
                                                                       "would exceed this wall time (at least one prove always runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--window-bits", type=int, default=0, help="MSM window override (0: chosen from the per-rank MSM size)")
    ap.add_argument("--no-verify", action="store_true", help="skip the post-run proof check (oracle verifier with the real pairing)")
    ap.add_argument("--save-proof", default=None, help="write the hashed proof, the verifier key and the public data to this JSON file "
                                                       "(checked afterwards on a CPU by tests/verify_saved_proof.py)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write the proof of the last step of each timed region as DIR/proof.npy (device-resident "
                         "instance) and DIR/proof_e2e.npy (host buffers): one float32 per proof byte.  Inputs and zk stream are seeded, so "
                         "two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md): one
    long-running `nvidia-smi -lms` process started before the warm-up (so its start-up cost never lands
    in a timed step); mark() brackets the timed region and only samples inside it are summarised."""
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, period_ms=250):
        self.lines = []
        self.t_lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", str(period_ms)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        self.t0 = self.t1 = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())
            self.t_lines.append(time.time())

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def close(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=3)
            except Exception:
                self.proc.kill()

    def summary(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        sm, mx, reasons = [], None, set()
        for t, line in zip(self.t_lines, self.lines):
            if self.t0 is None or self.t1 is None or not (self.t0 <= t <= self.t1 + 0.3):
                continue
            parts = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(parts[1]))
                mx = float(parts[2])
            except Exception:
                continue
            for n, v in zip(names, parts[3:]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_baseline(args, log_n, repeats=1, time_budget_s=None):
    """Oracle C++ restatement of the reference prover (oracle/cport) on this box's host cores."""
    try:
        from oracle import cport
        return cport.prover_baseline(args.curve, args.pc, log_n, repeats=repeats, time_budget_s=time_budget_s)
    except Exception as e:  # the baseline is reported, never required for the GPU number
        return {"value": None, "unit": "constraints/s", "cores": 0, "kind": "port", "sample": f"unavailable: {e}"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU prover path (its C++/OpenMP restatement, oracle/cport -- the Rust
    reference cannot be built in this image) on the SAME configuration as the GPU arm: Marlin::prove of DummyCircuit
    2^log_n, all usable host threads, timed like benches/bench.rs:92-107 (prove only; SRS and index are set-up).  One
    2^20 prove takes about a minute of CPU time, so the run is bounded by --ref-budget-s: `steps` reports the proves
    actually timed (at least 1, at most --steps), `steps_requested` what the command line asked for."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.time()
    log_n = args.ref_log_n if args.ref_log_n else args.log_n
    base = cpu_baseline(args, log_n, repeats=max(1, args.steps), time_budget_s=args.ref_budget_s)
    v = base.get("value")
    n = 1 << log_n
    steps_run = base.get("steps_run", 0)
    line = {
        "impl": "reference", "metric": "prover_constraints_per_sec", "value": v, "unit": "constraints/s", "n_gpus": args.gpus,
        "steps": steps_run, "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
        "ms_per_step": (1000.0 * n / v) if v else None, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u64-limb modular integers (Fr 255-bit, Fq 381-bit)", "data": "synthetic",
        "config": {"workload": f"Marlin::prove, DummyCircuit 2^{log_n} constraints (|H|=2^{log_n}, |K|=2^{log_n + 2}), "
                               f"{args.curve}, {args.pc}, SimpleHashFiatShamirRng<Blake2s,ChaChaRng>",
                   "same_config_as_gpu_arm": log_n == args.log_n,
                   "timing": f"wall clock around each prove; {steps_run} of {args.steps} requested steps fit the {args.ref_budget_s:.0f} s "
                             "budget (no warm-up steps: a CPU prove has no cold-start effect worth a minute of budget)"},
        "cpu_baseline": dict(base or {}, value=v),
        "e2e": {"value": v, "unit": "constraints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    print(json.dumps(line))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
        return
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import torch
    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from marlin_b200 import api, r1cs
    n = 1 << args.log_n
    m = api.Marlin(args.curve, args.pc, device=local_rank)
    if world > 1:
        from marlin_b200 import multi
        multi.attach(m.ctx, dist, rank, world)
    cid = m.curve_id
    a, b = 0x1234567890abcdef1234567890abcdef, 0xfedcba0987654321fedcba0987654321
    circ = r1cs.dummy_circuit(cid, a, b, 10, n)
    t0 = time.time()
    srs = m.universal_setup(n, n, 3 * n, beta=0x5eed5eed5eed5eed5eed5eed, gamma=7, degree_bounds=(n - 2, 4 * n - 2),
                            window_bits=args.window_bits)
    pk = m.index(srs, circ)
    setup_s = time.time() - t0
    m.stage(pk, circ)
    zk = api.ZkRng.test_rng()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    clocks = ClockSampler(local_rank)
    for _ in range(max(args.warmup, 3)):
        m.prove(pk, None, zk)
    barrier()
    # ---- timed region 1: device-resident inputs (value), per-kernel events on ---------------------
    launches0 = m.ctx.launches()
    m.ctx.profile(True)
    dev_ms = []
    clocks.begin()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proof_dev = m.prove(pk, None, zk)
        dev_ms.append(pk.timings()["Marlin::Prover"])  # CUDA events on the library's stream
    barrier()
    wall = time.perf_counter() - t0
    clocks.end()
    kern = m.ctx.profile_report()
    m.ctx.profile(False)
    launches = m.ctx.launches() - launches0
    phases = pk.timings()
    # ---- timed region 2: end to end through the public API with host buffers ------------------------
    # the instance lives in PINNED host memory (torch allocates it; the library copies from it every step)
    pinned_inst = torch.from_numpy(circ.instance.view("int64")).pin_memory()
    pinned_wit = torch.from_numpy(circ.witness.view("int64")).pin_memory()
    circ.instance = pinned_inst.numpy().view("uint64")
    circ.witness = pinned_wit.numpy().view("uint64")
    barrier()
    t0 = time.perf_counter()
    proof = b""
    for _ in range(args.steps):
        proof = m.prove(pk, circ, zk)
    barrier()
    wall_e2e = time.perf_counter() - t0
    clocks.close()
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, blob in (("proof", proof_dev), ("proof_e2e", proof)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), np.frombuffer(blob, dtype=np.uint8).astype(np.float32))
    # outside every timed region: a proof from a fresh zk stream, hashed, so that runs with different window sizes,
    # GPU counts or library builds can be compared byte for byte
    import hashlib
    proof_chk = m.prove(pk, circ, api.ZkRng.test_rng())
    proof_sha = hashlib.sha256(proof_chk).hexdigest()
    # ---- checker (outside every timed region; rank 0): the proof must be accepted by the oracle's restatement of
    # Marlin::verify -- trapdoor identity AND the reference's real product of pairings -- rejected for a wrong public input,
    # and equal to the pinned 1-GPU proof of the same instance where one is recorded (tests/golden/bench_proof_hashes.json).
    proof_check, proof_verified, proof_matches = None, None, None
    if rank == 0:
        from marlin_b200 import fields
        blob = {"curve": args.curve, "pc": args.pc, "log_n": args.log_n, "n_gpus": world, "max_degree": int(srs.max_degree),
                "beta": 0x5eed5eed5eed5eed5eed5eed, "gamma": 7, "public_input": [str(a * b % fields.FR_MODULUS[cid])],
                "proof_hex": proof_chk.hex(), "vk_hex": bytes(pk.vk_bytes).hex(), "proof_sha256": proof_sha}
        if args.save_proof:
            with open(args.save_proof, "w") as f:
                json.dump(blob, f)
        try:
            with open(os.path.join(ROOT, "tests", "golden", "bench_proof_hashes.json")) as f:
                pinned = json.load(f).get(f"{args.curve}/{args.pc}/{args.log_n}")
            proof_matches = (pinned == proof_sha) if pinned else None
        except Exception:
            pass
        if not args.no_verify:
            try:
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                import verify_saved_proof
                t_v = time.time()
                proof_check = verify_saved_proof.verify_blob(blob, use_pairing=True)
                proof_check["seconds"] = time.time() - t_v
                proof_verified = bool(proof_check["ok"])
            except Exception as e:
                proof_check = {"error": repr(e)}
                proof_verified = False

    ms_step = sum(dev_ms) / len(dev_ms)
    if dist is not None:  # max over ranks
        t = torch.tensor([ms_step, wall, wall_e2e], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, wall, wall_e2e = (float(x) for x in t.tolist())
    value = n / (ms_step / 1e3)
    e2e_value = n * args.steps / wall_e2e
    peaks, peak_kind = measured_peaks()
    zero = {"ms": 0.0, "units": 0.0, "launches": 0}
    acc = kern.get("msm_accumulate_kernel", zero)
    lev = kern.get("msm_affine_levels", zero)
    pair_bytes = 128 if args.curve == "bls12_381" else 96
    # The dominant kernels are the MSM bucket pass: (3 batched-affine level kernels, where the MSM is large enough)
    # + the XYZZ accumulate kernel on what is left.  One "launch" below = the bucket pass of one MSM.
    bucket_ms = acc["ms"] + lev["ms"]
    achieved = (acc["units"] * pair_bytes / (bucket_ms / 1e3) / 1e9) if bucket_ms else None
    from marlin_b200 import _lib as _plib
    win_bits = int(_plib.lib().b2m_srs_window_bits(srs.handle))
    aff_levels = int(_plib.lib().b2m_srs_affine_levels(srs.handle))
    scalar_bits = 255 if args.curve == "bls12_381" else 254
    msm_windows, mul_peak = (scalar_bits + win_bits) // win_bits, None  # signed c-bit windows per scalar (c = 20 -> 13)
    try:
        with open(os.path.join(ROOT, "profiles", "r02_microbench_int_alu.json")) as f:
            mb = json.load(f)
        mul_peak = max(v for k, v in mb.items() if k.startswith("fq_mul")) if args.curve == "bls12_381" else None
    except Exception:
        pass
    # field multiplications the bucket pass performs: an affine addition with a shared inversion is 6, an XYZZ mixed
    # addition 10; L levels leave 1/2^L of the references to the XYZZ kernel
    share = 0.5 ** aff_levels
    muls = msm_windows * (lev["units"] * ((1 - share) * 6 + share * 10) + (acc["units"] - lev["units"]) * 10)
    traffic = None  # DRAM bytes per launch from the committed `ncu --set full` capture of THIS round's kernels (profiles/), scaled to this run's mean launch
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as f:
            tr = json.load(f)
        if args.curve == "bls12_381" and acc["launches"]:
            per_pair = (tr["levels"]["dram_bytes_per_pair"] + tr["accumulate_after_levels"]["dram_bytes_per_pair"]) if lev["launches"] else tr["dram_bytes_per_pair"]
            traffic = per_pair * acc["units"] / acc["launches"]
    except Exception:
        pass
    line = {
        "metric": "prover_constraints_per_sec", "value": value, "unit": "constraints/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32-limb modular integers (Fr 255-bit, Fq 381-bit)", "data": "synthetic",
        "config": {"workload": f"Marlin::prove, DummyCircuit 2^{args.log_n} constraints (|H|=2^{args.log_n}, |K|=2^{args.log_n + 2}), "
                               f"{args.curve}, {args.pc}, SimpleHashFiatShamirRng<Blake2s,ChaChaRng>",
                   "timing": "CUDA events on the library stream around each prove; working set (SRS tables + index + polynomials, "
                             "> 7 GB) exceeds L2, no flush needed",
                   "msm_window_bits": win_bits, "parallelism": f"msm-shard x{world}" if world > 1 else "single"},
        "wall_ms_per_step": 1e3 * wall / args.steps,
        "gpu_launches": launches // args.steps,
        "e2e": {"value": e2e_value, "unit": "constraints/s", "h2d_bytes_per_step": int(circ.instance.nbytes + circ.witness.nbytes),
                "d2h_bytes_per_step": len(proof) + 15 * 96, "host_memory": "pinned"},
        "clocks": clocks.summary(),
        "roofline": {"bound": "hbm", "kernel": ("MSM bucket pass: %d batched-affine level kernels (fused level 0, split levels >= 1) + msm_accumulate_kernel" % aff_levels) if lev["launches"]
                     else "msm_accumulate_kernel", "achieved": achieved, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                     "frac": (achieved / peaks["hbm_gbs"]) if achieved else None, "traffic": traffic, "peak_source": peak_kind,
                     "algorithmic_bytes_per_launch": (acc["units"] * pair_bytes / acc["launches"]) if acc["launches"] else None,
                     "algorithmic_bytes_per_pair": pair_bytes, "launch": "the bucket pass of one MSM (mean over the proof's MSMs)",
                     "note": "bound by the 32-bit integer multiplier, not by HBM (roofline_int_alu; DESIGN.md Rooflines); traffic = "
                             "level + accumulate kernels of one 2^22-pair MSM (profiles/r02_ncu_level_accumulate.md)"},
        # the meaningful roofline of these kernels: Fq multiplications per second against the whole-chip
        # integer-multiply microbenchmark (profiles/r02_microbench_int_alu.json, tools/microbench.cu)
        "roofline_int_alu": {"kernel": "MSM bucket pass", "unit": "G Fq multiplications/s",
                             "achieved": (muls / (bucket_ms / 1e3) / 1e9) if bucket_ms else None,
                             "peak": mul_peak, "frac": (muls / (bucket_ms / 1e3) / 1e9 / mul_peak) if bucket_ms and mul_peak else None,
                             "affine_levels": aff_levels, "muls_per_affine_add": 6, "muls_per_xyzz_add": 10,
                             "bucket_additions_per_s_G": (acc["units"] * msm_windows / (bucket_ms / 1e3) / 1e9) if bucket_ms else None,
                             "peak_source": "tools/microbench.cu fq_mul (measured on this pool's B200)"},
        "msm_bucket_pass_ms_per_step": bucket_ms / args.steps if bucket_ms else None,
        "kernels": kern, "phases_ms": phases, "dev_ms_steps": dev_ms, "setup_s": setup_s, "proof_bytes": len(proof), "proof_sha256": proof_sha,
        "proof_verified": proof_verified, "proof_matches_pinned_1gpu_hash": proof_matches, "proof_check": proof_check,
    }
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, args.cpu_log_n, repeats=2, time_budget_s=30)
        print(json.dumps(line))
    pk.close()
    srs.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
