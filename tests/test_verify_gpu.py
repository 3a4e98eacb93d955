"""GPU: `Marlin.verify` / `Marlin.batch_verify` (b2m_verifier, b2m_verify) -- acceptance of honest proofs for both curves and PC
schemes, rejection of a wrong public input [reference src/test.rs:158-161], the committed golden proofs and replay kit, exact
verdicts for tampered proofs inside a batch, and one pairing product for an all-good batch."""
import hashlib
import json
import os
import random

import pytest

from marlin_b200 import _lib, api, r1cs as gr1cs
from oracle import ec, kzg, r1cs as or1cs
from oracle import rng as orng
from oracle import transcript as T
from oracle.params import BLS12_381, CURVES

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ACC, REJ, MAL = _lib.VERDICT_ACCEPT, _lib.VERDICT_REJECT, _lib.VERDICT_MALFORMED
REF_SHAPES = [(100, 25), (26, 25), (25, 100), (25, 26), (25, 25)]


@pytest.fixture(scope="module")
def gctx(b2m_ctx):
    c = api.Context.__new__(api.Context)
    c.handle = b2m_ctx
    return c


def pow2(n):
    s = 1
    while s < n:
        s *= 2
    return s


def build(gctx, curve, scheme, kind, nc, nv):
    """SRS (trapdoor), index and verifier key for a test or dummy circuit; returns (m, srs, pk, vk, circuit, public input)."""
    cid = 0 if curve is BLS12_381 else 1
    f = curve.fr
    rng = orng.test_rng()
    a, b = orng.field_rand(f, rng), orng.field_rand(f, rng)
    if kind == "test":
        ocirc, gcirc, pub = or1cs.test_circuit(f, a, b, nc, nv), gr1cs.test_circuit(cid, a, b, nc, nv), [a * b % f.p, a * b * b % f.p]
    else:
        ocirc, gcirc, pub = or1cs.dummy_circuit(f, a, b, nv, nc), gr1cs.dummy_circuit(cid, a, b, nv, nc), [a * b % f.p]
    cs = or1cs.synthesize(f, ocirc)
    am, bm, cm = cs.to_matrices()
    nnz = sum(len({i for _, i in ra} | {i for _, i in rb} | {i for _, i in rc}) for ra, rb, rc in zip(am, bm, cm))
    n = max(cs.num_constraints, len(cs.instance) + len(cs.witness))
    m = api.Marlin(curve.name, scheme, ctx=gctx)
    md = api.max_degree(n, n, nnz)
    srs = m.srs_from_trapdoor(md, beta=0x1234567, gamma=11, degree_bounds=(pow2(n) - 2, pow2(nnz) - 2))
    pk = m.index(srs, gcirc)
    vk = m.verifier_key(pk)
    return m, srs, pk, vk, gcirc, pub


def close(*objs):
    for o in objs:
        o.close()


CASES = ([("bls12_381", s, "test", nc, nv) for s in ("marlin_kzg10", "sonic_kzg10") for nc, nv in REF_SHAPES] +
         [(c, s, "dummy", 1 << k, 10) for c in ("bls12_381", "bn254") for s in ("marlin_kzg10", "sonic_kzg10") for k in (4, 8, 12)] +
         [("bn254", s, "test", 26, 25) for s in ("marlin_kzg10", "sonic_kzg10")])


@pytest.mark.parametrize("curve_name,scheme,kind,nc,nv", CASES, ids=lambda v: str(v))
def test_accepts_honest_proofs_and_rejects_wrong_input(gctx, curve_name, scheme, kind, nc, nv):
    curve = CURVES[curve_name]
    m, srs, pk, vk, circ, pub = build(gctx, curve, scheme, kind, nc, nv)
    try:
        zk = api.ZkRng.test_rng()
        p1, p2 = m.prove(pk, circ, zk), m.prove(pk, circ, zk)
        assert m.verify(vk, pub, p1)
        assert m.batch_verify(vk, [(pub, p1), (pub, p2)]) == [True, True]
        bad = [(pub[0] + 1) % curve.fr.p] + pub[1:]
        assert not m.verify(vk, bad, p1)
        assert m.last_verdicts == [REJ]
    finally:
        close(vk, pk, srs)


def _golden_cases():
    with open(os.path.join(HERE, "golden", "marlin_proofs.json")) as fh:
        return json.load(fh)["cases"]


@pytest.mark.parametrize("case", _golden_cases(), ids=lambda c: c["name"])
def test_golden_proofs_accepted(gctx, case):
    """The committed oracle proofs, with the verifier key rebuilt from the generator's parameters (tests/tests_golden.py)."""
    import tests_golden as tg
    curve = CURVES[case["curve"]]
    _, a, b, ocirc, pub = tg.case_inputs(case)
    cid = 0 if case["curve"] == "bls12_381" else 1
    scheme = "marlin_kzg10" if case["scheme"] == kzg.MARLIN else "sonic_kzg10"
    m = api.Marlin(case["curve"], scheme, ctx=gctx)
    g = ec.scalar_mul(curve, tg.G_SCALAR, curve.g)
    circ = gr1cs.test_circuit(cid, a, b, case["nc"], case["nv"]) if case["circuit"] == "test" else gr1cs.dummy_circuit(cid, a, b, case["nv"], case["nc"])
    cs = or1cs.synthesize(curve.fr, ocirc)
    am, bm, cm = cs.to_matrices()
    nnz = sum(len({i for _, i in ra} | {i for _, i in rb} | {i for _, i in rc}) for ra, rb, rc in zip(am, bm, cm))
    srs = m.srs_from_trapdoor(case["srs_max_degree"], beta=tg.BETA, g=g, gamma=tg.GAMMA,
                              degree_bounds=[pow2(circ.num_constraints) - 2, pow2(nnz) - 2])
    pk = m.index(srs, circ)
    vk = m.verifier_key(pk)
    try:
        assert hashlib.sha256(pk.vk_bytes).hexdigest() == case["vk_sha256"]
        proof = bytes.fromhex(case["proof_hex"])
        assert m.verify(vk, pub, proof)
        assert not m.verify(vk, [(pub[0] + 1) % curve.fr.p] + pub[1:], proof)
    finally:
        close(vk, pk, srs)


@pytest.mark.parametrize("scheme", ["marlin_kzg10", "sonic_kzg10"])
def test_replay_kit_from_public_files(gctx, scheme):
    kit = os.path.join(HERE, "golden", "replay_kit")
    meta = json.load(open(os.path.join(kit, "meta.json")))
    m = api.Marlin("bls12_381", scheme, ctx=gctx)
    vk = m.verifier_key_from_files(os.path.join(kit, "srs.bin"), open(os.path.join(kit, f"{scheme}_index_vk_tobytes.bin"), "rb").read())
    try:
        proof = open(os.path.join(kit, f"{scheme}_proof.bin"), "rb").read()
        pub = [int(x) for x in meta["public_input"]]
        assert m.verify(vk, pub, proof)
        assert not m.verify(vk, [pub[0] + 1], proof)
    finally:
        vk.close()


# ---- tampering -------------------------------------------------------------------------------------------------
def layout(proof, nb, marlin):
    """offsets of the fields of a serialized proof (the layout of oracle/marlin.py serialize_proof)"""
    off = 8
    comms, shifted = [], {}
    for count in (4, 3, 2):
        off += 8
        for _ in range(count):
            comms.append(off)
            off += nb
            if marlin:
                flag = proof[off]
                off += 1
                if flag:
                    shifted[len(comms) - 1] = off - 1
                    off += nb
    off += 8
    evals = off
    off += 4 * 32 + 8 + 3 + 8
    w, rv = [], []
    for _ in range(2):
        w.append(off)
        off += nb
        rv.append(off)
        off += 1 + (32 if proof[off] else 0)
    return {"comms": comms, "shifted": shifted, "evals": evals, "w": w, "rv": rv}


def tampered(curve, proof, marlin):
    """[(name, bytes, expected verdict)]"""
    nb, r, q = curve.fq.nbytes, curve.fr.p, curve.fq.p
    L = layout(proof, nb, marlin)
    out = []

    def put(b, at, data):
        b = bytearray(b)
        b[at:at + len(data)] = data
        return bytes(b)

    e0 = int.from_bytes(proof[L["evals"]:L["evals"] + 32], "little")
    out.append(("eval+1", put(proof, L["evals"], ((e0 + 1) % r).to_bytes(32, "little")), REJ))
    c0, c1 = L["comms"][0], L["comms"][1]
    out.append(("swap", put(put(proof, c0, proof[c1:c1 + nb]), c1, proof[c0:c0 + nb]), REJ))
    out.append(("other W", put(proof, L["w"][0], T.g1_compressed(curve, ec.scalar_mul(curve, 7, curve.g))), REJ))
    rv = L["rv"][0]
    if proof[rv]:
        v = int.from_bytes(proof[rv + 1:rv + 33], "little")
        out.append(("random_v+1", put(proof, rv + 1, ((v + 1) % r).to_bytes(32, "little")), REJ))
        out.append(("random_v dropped", proof[:rv] + b"\x00" + proof[rv + 33:], REJ))
    if marlin:
        i, flag = next(iter(L["shifted"].items()))
        out.append(("shifted dropped", proof[:flag] + b"\x00" + proof[flag + 1 + nb:], MAL))
    out.append(("eval >= r", put(proof, L["evals"], (r + 1).to_bytes(32, "little")), MAL))
    out.append(("x >= q", put(proof, c0, q.to_bytes(nb, "little")), MAL))
    x = 1
    while pow((x ** 3 + curve.b) % q, (q - 1) // 2, q) == 1:
        x += 1
    out.append(("non-residue", put(proof, c0, x.to_bytes(nb, "little")), MAL))
    if curve is BLS12_381:
        x = 0
        while pow((x ** 3 + 4) % q, (q - 1) // 2, q) != 1:
            x += 1
        out.append(("off subgroup", put(proof, c0, x.to_bytes(nb, "little")), MAL))
    out.append(("infinity", put(proof, c0, T.g1_compressed(curve, None)), REJ))
    out.append(("both flags", put(proof, c0 + nb - 1, bytes([proof[c0 + nb - 1] | 0xc0])), MAL))
    out.append(("truncated", proof[:-1], MAL))
    out.append(("extended", proof + b"\x00", MAL))
    return out


@pytest.mark.parametrize("curve_name,scheme", [("bls12_381", "marlin_kzg10"), ("bls12_381", "sonic_kzg10"), ("bn254", "marlin_kzg10")])
def test_tampered_proofs_exact_verdicts_in_a_batch(gctx, curve_name, scheme):
    curve = CURVES[curve_name]
    m, srs, pk, vk, circ, pub = build(gctx, curve, scheme, "dummy", 64, 10)
    try:
        zk = api.ZkRng.test_rng()
        good = [m.prove(pk, circ, zk) for _ in range(3)]
        bad = tampered(curve, good[0], scheme == "marlin_kzg10")
        items, want = [], []
        for k, (name, data, verdict) in enumerate(bad):
            items.append((pub, good[k % 3]))
            want.append(ACC)
            items.append((pub, data))
            want.append(verdict)
        m.batch_verify(vk, items, api.ZkRng(bytes(32)))
        got = m.last_verdicts
        names = [n for n, _, _ in bad]
        assert got == want, list(zip(["good", "bad"] * len(bad), [x for n in names for x in ("-", n)], want, got))
    finally:
        close(vk, pk, srs)


def test_batch_of_64_one_pairing_and_seed_independent(gctx):
    curve = BLS12_381
    m, srs, pk, vk, circ, pub = build(gctx, curve, "marlin_kzg10", "dummy", 256, 10)
    try:
        zk = api.ZkRng.test_rng()
        proofs = [m.prove(pk, circ, zk) for _ in range(4)]
        items = [(pub, proofs[i % 4]) for i in range(64)]
        gctx.profile(True)
        assert m.batch_verify(vk, items, api.ZkRng(bytes(32))) == [True] * 64
        rep = gctx.profile_report()
        gctx.profile(False)
        assert rep["verify_pairing"]["launches"] == 1 and rep["verify_pairing"]["units"] == 1
        t = vk.timings()
        assert set(t) >= {"decode", "transcript", "scalars", "combine", "fold", "pairing"}
        bad_at = {3, 17, 40, 63}
        rnd = random.Random(5)
        items2 = list(items)
        for i in bad_at:
            items2[i] = ([(pub[0] + rnd.randrange(1, 100))], proofs[i % 4]) if i % 2 else (pub, proofs[i % 4][:-1])
        want = [i not in bad_at for i in range(64)]
        v1 = m.batch_verify(vk, items2, api.ZkRng(bytes(32)))
        v2 = m.batch_verify(vk, items2, api.ZkRng(bytes([7] * 32)))
        assert v1 == want and v2 == want
        assert [m.verify(vk, p, pr) for p, pr in items2] == want
    finally:
        close(vk, pk, srs)



def test_full_size_bench_proof_accepted(gctx):
    """The 2^20-constraint BLS12-381 MarlinKZG10 proof of bench.py's configuration (same circuit, SRS trapdoor and zk stream)."""
    from marlin_b200 import fields
    n = 1 << 20
    m = api.Marlin("bls12_381", "marlin_kzg10", ctx=gctx)
    a, b = 0x1234567890abcdef1234567890abcdef, 0xfedcba0987654321fedcba0987654321
    circ = gr1cs.dummy_circuit(0, a, b, 10, n)
    srs = m.universal_setup(n, n, 3 * n, beta=0x5eed5eed5eed5eed5eed5eed, gamma=7, degree_bounds=(n - 2, 4 * n - 2))
    pk = m.index(srs, circ)
    vk = m.verifier_key(pk)
    try:
        proof = m.prove(pk, circ, api.ZkRng.test_rng())
        pub = [a * b % fields.FR_MODULUS[0]]
        assert m.verify(vk, pub, proof)
        assert not m.verify(vk, [pub[0] + 1], proof)
    finally:
        close(vk, pk, srs)
