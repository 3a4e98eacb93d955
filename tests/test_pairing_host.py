"""CPU: the pairing tower and optimal ate pairing (csrc/pairing.cuh), the compressed-point decoder and the linear-combination
coefficients (csrc/verify_core.cuh), compiled for the host and checked against the Python oracle.

The oracle's Fq12 is the single extension Fq[w]/(w^12 - 2 alpha w^6 + alpha^2 + 1) with w^6 = xi = alpha + u (oracle/pairing.py);
the tower's w is the same w and v = w^2, so tower element sum (a_ij + b_ij u) v^j w^i maps linearly onto it.  The optimal ate
pairing reference below runs its Miller loop over that untwisted E(Fq12) representation and exponentiates by (q^12 - 1) / r
directly; pairing.cuh's final exponentiation computes the power m (q^12 - 1) / r with m = 3 for BLS12-381 and 1 for BN254."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import ec, kzg, marlin as omarlin, pairing, r1cs as or1cs, rng as orng
from oracle.params import BLS12_381, BN254
from test_srs_files import Fq2Ref

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "host", "libpairing_host.so")
CSRC = os.path.join(HERE, "..", "marlin_b200", "csrc")

CURVES = [(0, BLS12_381), (1, BN254)]
IDS = ["bls12_381", "bn254"]
M = {0: 3, 1: 1}
ATE_LOOP = {0: 0xd201000000010000, 1: 6 * 4965661367192848881 + 2}
G2_GEN = {  # the standard generators on the twist (x.c0, x.c1, y.c0, y.c1), as in csrc/b2m_capi.cu
    0: (0x024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8,
        0x13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e,
        0x0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801,
        0x0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be),
    1: (0x1800deef121f1e76426a00665e5c4479674322d4f75edadd46debd5cd992f6ed,
        0x198e9393920d483a7260bfb731fb5d25f1aa493335a9e71297e485b7aef312c2,
        0x12c85ea5db8c6deb4aab71808dcb408fe3d1e7690c43d37b4ce6cc0166fa7daa,
        0x090689d0585ff075ec9e99ad690c3395bc4b313370b38ef355acdadcd122975b),
}


@pytest.fixture(scope="module")
def hostlib():
    src = os.path.join(HERE, "host", "pairing_host_shim.cpp")
    deps = [src] + [os.path.join(CSRC, h) for h in ("field.cuh", "curve.cuh", "pairing.cuh", "pairing_params.h", "verify_core.cuh")]
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O1", "-DB2M_HOST_LIGHT_INLINE", "-shared", "-fPIC", "-x", "c++", src, "-o", SO])
    return ctypes.CDLL(SO)


def nlimbs(curve):
    return 12 if curve.fq.p.bit_length() > 256 else 8


def to_limbs(vals, n, p, mont=True):
    R = 1 << (32 * n)
    out = []
    for v in vals:
        m = v * R % p if mont else v
        out += [(m >> (32 * i)) & 0xffffffff for i in range(n)]
    return (ctypes.c_uint32 * len(out))(*out)


def from_limbs(arr, count, n, p):
    Rinv = pow(1 << (32 * n), -1, p)
    return [sum(int(arr[k * n + i]) << (32 * i) for i in range(n)) * Rinv % p for k in range(count)]


def tower_to_oracle(eng, t):
    """12 tower coefficients (c_i.c_j.c_k order) -> oracle Fq12"""
    c = [0] * 12
    for i in range(2):
        for j in range(3):
            a, b = t[6 * i + 2 * j], t[6 * i + 2 * j + 1]
            k = i + 2 * j
            c[k] += a - eng.alpha * b
            c[k + 6] += b
    return eng.Fq12(c)


def fq12_call(lib, cid, curve, op, a, b=None, k=0):
    n = nlimbs(curve)
    p = curve.fq.p
    out = (ctypes.c_uint32 * (12 * n))()
    lib.fq12_op(cid, op, k, to_limbs(a, n, p), to_limbs(b or [0] * 12, n, p), out)
    return from_limbs(out, 12, n, p)


# ---- the reference optimal ate pairing over E(Fq12) ----------------------------------------------------------------
def ate(eng, cid, Pt, Q):
    Fq12 = eng.Fq12
    xp, yp = Fq12.from_fq(Pt[0]), Fq12.from_fq(Pt[1])

    def line(T, S):
        x1, y1 = T
        if S == T:
            lam = x1.square().scale(3) * y1.scale(2).inv()
        else:
            lam = (S[1] - y1) * (S[0] - x1).inv()
        return (yp - y1) - lam * (xp - x1)

    f, T = Fq12.one(), Q
    for bit in bin(ATE_LOOP[cid])[3:]:
        f = f.square() * line(T, T)
        T = eng.e12_add(T, T)
        if bit == "1":
            f = f * line(T, Q)
            T = eng.e12_add(T, Q)
    if cid == 0:  # x < 0
        f = f.inv()
    else:  # two Frobenius lines: + pi(Q), - pi^2(Q)
        q1 = (Q[0].pow(eng.P), Q[1].pow(eng.P))
        q2 = (q1[0].pow(eng.P), -(q1[1].pow(eng.P)))
        f = f * line(T, q1)
        T = eng.e12_add(T, q1)
        f = f * line(T, q2)
    return f.pow(eng.final_exp)


def g2_point(cid, curve, k):
    f2 = Fq2Ref(curve.fq.p)
    g = G2_GEN[cid]
    return f2.smul(k, ((g[0], g[1]), (g[2], g[3])))


def run_pairing(lib, cid, curve, pairs, final_exp=True):
    n = nlimbs(curve)
    p = curve.fq.p
    g1, g2, inf = [], [], []
    for P, Q in pairs:
        inf.append(1 if P is None else 0)
        g1 += [0, 0] if P is None else [P[0], P[1]]
        g2 += [Q[0][0], Q[0][1], Q[1][0], Q[1][1]]
    out = (ctypes.c_uint32 * (12 * n))()
    lib.pairing_product(cid, len(pairs), to_limbs(g1, n, p), to_limbs(g2, n, p), (ctypes.c_uint8 * len(inf))(*inf), 1 if final_exp else 0, out)
    return from_limbs(out, 12, n, p)


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_tower_matches_oracle(hostlib, cid, curve):
    eng = pairing.for_curve(curve)
    p = curve.fq.p
    rnd = random.Random(100 + cid)
    for _ in range(3):
        a = [rnd.randrange(p) for _ in range(12)]
        b = [rnd.randrange(p) for _ in range(12)]
        A, B = tower_to_oracle(eng, a), tower_to_oracle(eng, b)
        assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 0, a, b)) == A * B
        assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 1, a)) == A * A
        assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 2, a)) * A == eng.Fq12.one()
        assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 5, a)) == A.pow(p ** 6)
        # sparse line products equal the dense product with the same sparse element
        sparse = [0] * 12
        pos = (0, 1, 4) if cid == 0 else (0, 3, 4)
        for k in pos:
            sparse[2 * k], sparse[2 * k + 1] = b[2 * k], b[2 * k + 1]
        assert fq12_call(hostlib, cid, curve, 6, a, sparse) == fq12_call(hostlib, cid, curve, 0, a, sparse)
    a = [rnd.randrange(p) for _ in range(12)]
    A = tower_to_oracle(eng, a)
    for k in (1, 2, 3):
        assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 3, a, k=k)) == A.pow(p ** k)


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_final_exponentiation_is_the_fixed_power(hostlib, cid, curve):
    eng = pairing.for_curve(curve)
    p = curve.fq.p
    rnd = random.Random(7 + cid)
    a = [rnd.randrange(p) for _ in range(12)]
    want = tower_to_oracle(eng, a).pow(M[cid] * eng.final_exp)
    assert tower_to_oracle(eng, fq12_call(hostlib, cid, curve, 4, a)) == want


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_pairing_value_matches_oracle_ate(hostlib, cid, curve):
    eng = pairing.for_curve(curve)
    rnd = random.Random(11 + cid)
    r = curve.fr.p
    a, b = rnd.randrange(1, r), rnd.randrange(1, r)
    P = ec.scalar_mul(curve, a, curve.g)
    Qt = g2_point(cid, curve, b)
    got = tower_to_oracle(eng, run_pairing(hostlib, cid, curve, [(P, Qt)]))
    want = ate(eng, cid, P, eng.untwist(*Qt))
    assert got == want.pow(M[cid])
    assert got != eng.Fq12.one()


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_pairing_bilinear_and_products(hostlib, cid, curve):
    eng = pairing.for_curve(curve)
    rnd = random.Random(21 + cid)
    r = curve.fr.p
    one = [1] + [0] * 11
    G, H = curve.g, g2_point(cid, curve, 1)
    e1 = tower_to_oracle(eng, run_pairing(hostlib, cid, curve, [(G, H)]))
    a, b = rnd.randrange(1, r), rnd.randrange(1, r)
    eab = tower_to_oracle(eng, run_pairing(hostlib, cid, curve, [(ec.scalar_mul(curve, a, G), g2_point(cid, curve, b))]))
    assert eab == e1.pow(a * b % r)
    assert e1.pow(r) == eng.Fq12.one()
    # e(aG, H) * e(-G, aH) = 1 with one final exponentiation; a point at infinity contributes 1
    prod = run_pairing(hostlib, cid, curve, [(ec.scalar_mul(curve, a, G), H), (ec.affine_neg(curve, G), g2_point(cid, curve, a)), (None, H)])
    assert prod == one
    bad = run_pairing(hostlib, cid, curve, [(ec.scalar_mul(curve, a, G), H), (ec.affine_neg(curve, G), g2_point(cid, curve, a + 1))])
    assert bad != one


def _compressed(curve, x, flags):
    nb = curve.fq.nbytes
    b = bytearray(x.to_bytes(nb, "little"))
    b[-1] |= flags
    return bytes(b)


def decode(lib, cid, curve, data):
    n = nlimbs(curve)
    out = (ctypes.c_uint32 * (2 * n))()
    st = lib.g1_decode(cid, (ctypes.c_uint8 * len(data))(*data), out)
    x, y = from_limbs(out, 2, n, curve.fq.p)
    return st, (None if x == 0 and y == 0 else (x, y))


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_decode_matches_oracle_and_rejects(hostlib, cid, curve):
    from oracle import transcript as T
    rnd = random.Random(31 + cid)
    q = curve.fq.p
    for _ in range(8):
        P = ec.scalar_mul(curve, rnd.randrange(1, curve.fr.p), curve.g)
        data = T.g1_compressed(curve, P)
        assert decode(hostlib, cid, curve, data) == (0, omarlin._g1_decompress(curve, data))
    assert decode(hostlib, cid, curve, T.g1_compressed(curve, None)) == (0, None)
    assert decode(hostlib, cid, curve, _compressed(curve, 0, 0xc0))[0] == 1                     # both flags
    assert decode(hostlib, cid, curve, _compressed(curve, q, 0))[0] == 2                        # x = q
    assert decode(hostlib, cid, curve, _compressed(curve, q + 5, 0x80))[0] == 2                 # x > q
    x = 1
    while pow((x ** 3 + curve.b) % q, (q - 1) // 2, q) == 1:
        x += 1
    assert decode(hostlib, cid, curve, _compressed(curve, x, 0))[0] == 3                        # non-residue
    if cid == 0:
        # a point on E(Fq) outside the r-torsion: smallest x with a square right-hand side, not cofactor-cleared
        x = 0
        while pow((x ** 3 + 4) % q, (q - 1) // 2, q) != 1:
            x += 1
        assert decode(hostlib, cid, curve, _compressed(curve, x, 0))[0] == 4


@pytest.mark.parametrize("cid,curve", CURVES, ids=IDS)
def test_lc_coefficients_reproduce_oracle(hostlib, cid, curve):
    """verify_core.cuh lc_coefficients, fed the challenges the oracle prover records, gives the oracle's LCs."""
    from oracle import ahp
    from oracle.poly import Domain, evaluate
    f = curve.fr
    rng = orng.test_rng()
    a, b = orng.field_rand(f, rng), orng.field_rand(f, rng)
    circ = or1cs.dummy_circuit(f, a, b, 10, 32)
    srs = omarlin.universal_setup(curve, 32, 32, 96, beta=0x1234567, g_scalar=1, gamma=7)
    eng = kzg.Engine(use_trapdoor=True)
    pk = omarlin.index(srs, circ, kzg.MARLIN, eng)
    proof = omarlin.prove(pk, circ, orng.test_rng(), eng)
    d = proof.debug
    public_input = [a * b % f.p]
    x_dom = Domain(f, len(public_input) + 1)
    formatted = [1] + public_input + [0] * (x_dom.size - 1 - len(public_input))
    n = 8
    ins = [d["alpha"], *d["eta"], d["beta"], d["gamma"]] + list(proof.evaluations)
    out = (ctypes.c_uint32 * (12 * n))()
    h, k = Domain(f, pk.index.info.num_constraints).size, Domain(f, pk.index.info.num_non_zero).size
    hostlib.lc_coeffs(cid, to_limbs(ins, n, f.p), to_limbs(formatted, n, f.p), len(formatted), h, k, out)
    got = from_limbs(out, 12, n, f.p)

    class VS:
        pass
    v = VS()
    v.domain_h, v.domain_k = Domain(f, pk.index.info.num_constraints), Domain(f, pk.index.info.num_non_zero)
    v.alpha, (v.eta_a, v.eta_b, v.eta_c), v.beta, v.gamma = d["alpha"], d["eta"], d["beta"], d["gamma"]
    ev = dict(zip(["g_1", "g_2", "t", "z_b"], proof.evaluations))
    lcs = {lc.label: lc for lc in ahp.construct_linear_combinations(f, public_input, lambda l, pt: ev[l], v)}

    def coeff(lc, label):
        return sum(c for c, t in lcs[lc].terms if t == label) % f.p

    want = [coeff("outer_sumcheck", "z_a"), coeff("outer_sumcheck", "w"), coeff("outer_sumcheck", "h_1"), coeff("outer_sumcheck", None),
            coeff("inner_sumcheck", "a_val"), coeff("inner_sumcheck", "b_val"), coeff("inner_sumcheck", "c_val"),
            coeff("inner_sumcheck", "row"), coeff("inner_sumcheck", "col"), coeff("inner_sumcheck", "row_col"),
            coeff("inner_sumcheck", "h_2"), coeff("inner_sumcheck", None)]
    assert coeff("outer_sumcheck", "mask_poly") == 1
    assert got == want
