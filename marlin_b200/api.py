"""Host-side mirror of the reference's public API for the accelerated path:
`Marlin::<F, PC, FS>::{universal_setup, index, prove}` [reference src/lib.rs:79-311] with
F in {BLS12-381 Fr, BN254 Fr}, PC in {MarlinKZG10, SonicKZG10}, FS = SimpleHashFiatShamirRng<Blake2s, ChaChaRng>.
Every call lands in libb2m.so (include/b2m.h); nothing here computes on the CPU beyond marshalling.

`Marlin::verify` [reference src/lib.rs:315-433] is `Marlin.verify` / `Marlin.batch_verify` against a device-resident
`VerifierKey` (b2m_verifier): compressed points are decoded and subgroup-checked on the GPU, the Fiat-Shamir transcripts are
replayed on host threads, and a whole batch is folded into one pairing product checked on the GPU.  Proofs are
`CanonicalSerialize` bytes, the same bytes the reference's `Marlin::verify` consumes.
"""
import ctypes
import json
import os
import struct

import numpy as np

from . import _lib, fields

PC_IDS = {"marlin_kzg10": _lib.PC_MARLIN_KZG10, "sonic_kzg10": _lib.PC_SONIC_KZG10}


class Context:
    """One GPU (b2m_ctx)."""

    def __init__(self, device=0):
        self.handle = ctypes.c_void_p()
        _lib.check(_lib.lib().b2m_ctx_create(device, ctypes.byref(self.handle)))

    def launches(self):
        return int(_lib.lib().b2m_ctx_launches(self.handle))

    def profile(self, enable=True):
        _lib.check(_lib.lib().b2m_ctx_profile(self.handle, 1 if enable else 0))

    def profile_report(self):
        buf = ctypes.create_string_buffer(1 << 16)
        _lib.check(_lib.lib().b2m_ctx_profile_report(self.handle, buf, 1 << 16))
        return json.loads(buf.value.decode() or "{}")

    def close(self):
        if self.handle:
            _lib.lib().b2m_ctx_destroy(self.handle)
            self.handle = None


class ZkRng:
    """The caller's `zk_rng` as a ChaCha stream position.  Like the reference, which makes the caller pass
    `zk_rng: &mut R` [reference src/lib.rs:154], there is no implicit fixed seed: `ZkRng()` seeds from
    os.urandom(32); the public `ark_std::test_rng()` stream (ChaCha12, fixed seed -- NOT zero-knowledge, every
    blinding value is predictable) is only available through the explicit `ZkRng.test_rng()` used by tests
    and the bench."""
    TEST_RNG_SEED = bytes([1, 0, 0, 0, 23, 0, 0, 0, 200, 1, 0, 0, 210, 30, 0, 0] + [0] * 16)

    def __init__(self, seed=None, rounds=12, word_pos=0):
        self.c = _lib.Rng()
        self.c.kind = rounds
        seed = os.urandom(32) if seed is None else bytes(seed)
        if len(seed) != 32:
            raise ValueError("ZkRng seed must be 32 bytes")
        ctypes.memmove(self.c.key, seed, 32)
        self.c.word_pos = word_pos

    @classmethod
    def test_rng(cls):
        """`ark_std::test_rng()`: rand 0.8 StdRng (ChaCha12) with the public fixed seed.  Tests / benchmarks only."""
        return cls(cls.TEST_RNG_SEED, 12, 0)

    @property
    def word_pos(self):
        return int(self.c.word_pos)


class CallbackRng:
    """Any other `RngCore` behind the C ABI (B2M_RNG_CALLBACK): `next_u64` is a Python callable returning the generator's next
    64-bit output; the library pulls every random value the reference would draw through it, in the reference's order."""

    def __init__(self, next_u64):
        self._fn = next_u64
        self._cb = _lib.NEXT_U64(lambda _state: int(self._fn()) & 0xFFFFFFFFFFFFFFFF)  # kept alive with the object
        self.c = _lib.Rng()
        self.c.kind = _lib.RNG_CALLBACK
        self.c.next_u64 = self._cb
        self.c.state = None

    @property
    def word_pos(self):
        return None


class CommitterKey:
    """`PC::CommitterKey` after `PC::trim` (b2m_ck): a validated view of the device-resident SRS."""

    def __init__(self, srs, handle, pc, supported_degree, hiding_bound, degree_bounds):
        self.srs, self.handle, self.pc = srs, handle, pc
        self.supported_degree, self.hiding_bound, self.degree_bounds = supported_degree, hiding_bound, sorted(set(degree_bounds))

    def shift_power(self, bound):
        """MarlinKZG10 verifier key entry for an enforced bound: powers_of_g[max_degree - bound] (affine limbs)."""
        lq = _lib.LIMBS[self.srs.curve_id][1]
        out = np.zeros(2 * lq, dtype=np.uint64)
        _lib.check(_lib.lib().b2m_ck_shift_power(self.handle, bound, _lib.ptr(out)))
        return out

    def close(self):
        if self.handle:
            _lib.lib().b2m_ck_destroy(self.handle)
            self.handle = None


class UniversalSRS:
    """`PC::UniversalParams`, device resident (b2m_srs): G1 powers + the gamma powers the PC needs."""

    def __init__(self, ctx, curve_id, handle, max_degree, powers_limbs, gamma_limbs=None, gamma_indices=None):
        self.ctx, self.curve_id, self.handle, self.max_degree = ctx, curve_id, handle, max_degree
        self.powers_limbs, self.gamma_limbs, self.gamma_indices = powers_limbs, gamma_limbs, gamma_indices
        self.trapdoor = None  # (beta, gamma) of an insecure test SRS made by universal_setup / srs_from_trapdoor
        self.g2 = None        # (h, beta_h, {index: neg power}) as ark-serialize bytes when loaded from / written to a file

    def save(self, path, degree_bounds=()):
        """Write the SRS as an ark-serialize file (marlin_b200/srsfile.py).  The G2 half -- h, beta h and SonicKZG10's
        beta^-(max_degree - d) h per enforced bound -- comes from the trapdoor of a test SRS, or from the file it was loaded from."""
        from . import srsfile
        L = _lib.lib()
        g1 = 2 * srsfile.fq_bytes(self.curve_id)
        n = self.max_degree + 1
        powers = np.zeros(n * g1, dtype=np.uint8)
        _lib.check(L.b2m_srs_export_g1(self.handle, 0, n, _lib.ptr(powers)))
        gam = np.zeros(len(self.gamma_indices) * g1, dtype=np.uint8)
        _lib.check(L.b2m_g1_to_uncompressed(self.ctx.handle, self.curve_id, _lib.ptr(np.ascontiguousarray(self.gamma_limbs)), len(self.gamma_indices),
                                            _lib.ptr(gam)))
        graw = gam.tobytes()
        gamma = {int(k): graw[i * g1:(i + 1) * g1] for i, k in enumerate(self.gamma_indices)}
        if self.trapdoor is not None:
            h, beta_h, neg = srsfile.g2_setup(self.curve_id, fields.FR_MODULUS[self.curve_id], self.trapdoor[0], self.max_degree, degree_bounds)
        elif self.g2 is not None:
            h, beta_h, neg = self.g2
        else:
            raise ValueError("this SRS has no G2 half (neither a trapdoor nor a source file)")
        srsfile.write_srs(path, self.curve_id, powers.tobytes(), gamma, h, beta_h, neg)

    def close(self):
        if self.handle:
            _lib.lib().b2m_srs_destroy(self.handle)
            self.handle = None


class IndexProverKey:
    def __init__(self, srs, handle, r1cs, pc):
        self.srs, self.handle, self.pc = srs, handle, pc
        self.num_constraints, self.num_variables = r1cs.num_constraints, r1cs.num_variables
        L = _lib.lib()
        n = ctypes.c_size_t(0)
        _lib.check(L.b2m_index_vk_bytes(handle, None, 0, ctypes.byref(n)))
        buf = (ctypes.c_uint8 * n.value)()
        _lib.check(L.b2m_index_vk_bytes(handle, buf, n.value, ctypes.byref(n)))
        self.vk_bytes = bytes(buf)
        lq = _lib.LIMBS[srs.curve_id][1]
        self.index_comms = np.zeros((6, 2 * lq), dtype=np.uint64)
        _lib.check(L.b2m_index_comms(handle, _lib.ptr(self.index_comms)))

    def timings(self):
        buf = ctypes.create_string_buffer(4096)
        _lib.check(_lib.lib().b2m_prove_timings(self.handle, buf, 4096))
        return json.loads(buf.value.decode() or "{}")

    def close(self):
        if self.handle:
            _lib.lib().b2m_index_destroy(self.handle)
            self.handle = None


class VerifierKey:
    """`Marlin::verify`'s key on the device (b2m_verifier): the index_vk ToBytes image, the six index commitments, g, gamma g,
    prepared h and beta h, and the enforced degree bounds with their shift powers (MarlinKZG10) or beta^-(D - d) h (SonicKZG10)."""

    def __init__(self, ctx, curve_id, pc, handle, vk_bytes):
        self.ctx, self.curve_id, self.pc, self.handle, self.vk_bytes = ctx, curve_id, pc, handle, vk_bytes

    def timings(self):
        """Per-stage times (ms) of the last verification with this key."""
        buf = ctypes.create_string_buffer(4096)
        _lib.check(_lib.lib().b2m_verify_timings(self.handle, buf, 4096))
        return json.loads(buf.value.decode() or "{}")

    def close(self):
        if self.handle:
            _lib.lib().b2m_verifier_destroy(self.handle)
            self.handle = None


def _pow2_at_least(n):
    s = 1
    while s < n:
        s *= 2
    return s


def _index_bounds(vk_bytes):
    """The degree bounds an index's proofs use: |H| - 2 (g_1) and |K| - 2 (g_2) [reference src/ahp/mod.rs get_degree_bounds]."""
    _nv, nc, nnz = struct.unpack_from("<QQQ", vk_bytes, 0)
    return sorted({_pow2_at_least(nc) - 2, _pow2_at_least(nnz) - 2})


def max_degree(num_constraints, num_variables, num_non_zero):
    """`AHPForR1CS::max_degree` [reference src/ahp/mod.rs:71-93]"""
    def p2(n):
        s = 1
        while s < n:
            s *= 2
        return s
    h = p2(max(num_variables, num_constraints))
    k = p2(num_non_zero)
    return max(2 * h + 1 - 2, 3 * h + 2 - 3, h, h, k - 1)


class Marlin:
    """`Marlin<F, PC, FS>` for one curve and PC scheme on one GPU."""

    def __init__(self, curve="bls12_381", pc="marlin_kzg10", device=0, ctx=None):
        self.curve_id = fields.CURVE_IDS[curve]
        self.pc = PC_IDS[pc]
        self.ctx = ctx or Context(device)

    # -- universal_setup ---------------------------------------------------------------------------
    def universal_setup(self, num_constraints, num_variables, num_non_zero, beta, g=None, gamma=7, degree_bounds=(),
                        window_bits=0):
        """[reference src/lib.rs:79-96] with an explicit trapdoor: an insecure test SRS exactly like the
        reference's `universal_setup(.., test_rng)`, generated on the GPU.  `degree_bounds`: bounds whose
        shifted gamma powers SonicKZG10 will need (ignored by MarlinKZG10)."""
        md = max_degree(num_constraints, num_variables, num_non_zero)
        return self.srs_from_trapdoor(md, beta, g, gamma, degree_bounds, window_bits)

    def srs_from_trapdoor(self, md, beta, g=None, gamma=7, degree_bounds=(), window_bits=0):
        L = _lib.lib()
        cid = self.curve_id
        lq = _lib.LIMBS[cid][1]
        g = g or fields.G1_GENERATOR[cid]
        r = fields.FR_MODULUS[cid]
        g_l = _lib.ints_to_limbs([fields.fq_to_mont(cid, g[0]), fields.fq_to_mont(cid, g[1])], lq).reshape(1, 2 * lq)
        beta_l = _lib.ints_to_limbs([beta % r], 4)
        powers = np.zeros((md + 1, 2 * lq), dtype=np.uint64)
        _lib.check(L.b2m_g1_powers(self.ctx.handle, cid, _lib.ptr(g_l), _lib.ptr(beta_l), md + 1, _lib.ptr(powers)))
        # gamma powers: gamma * beta^i * g = one-term MSMs of the G1 powers
        idx = [0, 1, 2]
        for d in sorted(set(degree_bounds)):
            idx += [md - d + i for i in range(3) if md - d + i <= md]
        idx = sorted(set(idx))
        # powers_of_gamma_g at the needed exponents: FixedBaseMSM(gamma_g, [beta^i]) with gamma_g = gamma * g
        gamma_g = np.zeros((1, 2 * lq), dtype=np.uint64)
        _lib.check(L.b2m_fixed_base_msm(self.ctx.handle, cid, _lib.ptr(g_l), _lib.ptr(_lib.ints_to_limbs([gamma % r], 4)), 1, _lib.ptr(gamma_g)))
        exps = _lib.ints_to_limbs([pow(beta % r, i, r) for i in idx], 4)
        gam = np.zeros((len(idx), 2 * lq), dtype=np.uint64)
        _lib.check(L.b2m_fixed_base_msm(self.ctx.handle, cid, _lib.ptr(gamma_g), _lib.ptr(exps), len(idx), _lib.ptr(gam)))
        srs = self.srs_from_points(powers, gam, idx, window_bits)
        srs.trapdoor = (beta % r, gamma % r)
        return srs

    def load_srs(self, path, window_bits=0):
        """Load an SRS file (marlin_b200/srsfile.py layout; `deserialize_unchecked` semantics: no subgroup check)."""
        from . import srsfile
        L = _lib.lib()
        d = srsfile.read_srs(path)
        if d["curve_id"] != self.curve_id:
            raise ValueError(f"{path} holds curve {d['curve_id']}, this Marlin instance is curve {self.curve_id}")
        lq = _lib.LIMBS[self.curve_id][1]
        g1 = 2 * srsfile.fq_bytes(self.curve_id)
        n = len(d["powers"]) // g1
        powers = np.zeros((n, 2 * lq), dtype=np.uint64)
        raw = np.frombuffer(d["powers"], dtype=np.uint8)
        _lib.check(L.b2m_g1_from_uncompressed(self.ctx.handle, self.curve_id, _lib.ptr(np.ascontiguousarray(raw)), n, _lib.ptr(powers)))
        idx = sorted(d["gamma"])
        graw = np.frombuffer(b"".join(d["gamma"][k] for k in idx), dtype=np.uint8)
        gam = np.zeros((len(idx), 2 * lq), dtype=np.uint64)
        _lib.check(L.b2m_g1_from_uncompressed(self.ctx.handle, self.curve_id, _lib.ptr(np.ascontiguousarray(graw)), len(idx), _lib.ptr(gam)))
        srs = self.srs_from_points(powers, gam, idx, window_bits)
        srs.g2 = (d["h"], d["beta_h"], d["neg_powers"])
        return srs

    def srs_from_points(self, powers_limbs, gamma_limbs, gamma_indices, window_bits=0):
        """Upload an existing SRS (affine Montgomery limbs, as ark-ff stores them)."""
        L = _lib.lib()
        h = ctypes.c_void_p()
        gi = np.asarray(gamma_indices, dtype=np.uint64)
        powers_limbs = np.ascontiguousarray(powers_limbs)
        gamma_limbs = np.ascontiguousarray(gamma_limbs)
        _lib.check(L.b2m_srs_create(self.ctx.handle, self.curve_id, _lib.ptr(powers_limbs), len(powers_limbs), _lib.ptr(gamma_limbs),
                                    _lib.ptr(gi), len(gi), window_bits, ctypes.byref(h)))
        return UniversalSRS(self.ctx, self.curve_id, h, len(powers_limbs) - 1, powers_limbs, gamma_limbs, [int(i) for i in gi])

    # -- PC::trim (Level 1) ---------------------------------------------------------------------------------
    def trim(self, srs, supported_degree, supported_hiding_bound, enforced_degree_bounds=()):
        """`PC::trim(pp, supported_degree, supported_hiding_bound, enforced_degree_bounds)` [reference src/lib.rs:112-121]
        -> CommitterKey (the verifier key's G1 part is read with CommitterKey.shift_power)."""
        L = _lib.lib()
        h = ctypes.c_void_p()
        b = np.asarray(sorted(enforced_degree_bounds), dtype=np.uint64)
        _lib.check(L.b2m_trim(srs.handle, self.pc, supported_degree, supported_hiding_bound, _lib.ptr(b) if len(b) else None, len(b),
                              ctypes.byref(h)))
        return CommitterKey(srs, h, self.pc, supported_degree, supported_hiding_bound, [int(x) for x in b])

    def open_combinations(self, ck, polys, rands, shifted_rands, lcs, query_set, points, challenge_limbs):
        """`PC::open_combinations` [reference src/lib.rs:292-302].  polys: (coeff limbs, degree_bound, hiding_bound) as for
        `commit`; rands / shifted_rands as returned by `commit`; lcs: list of term lists [(coeff Montgomery limbs (4,), poly index
        or None for the constant term)], in label order; query_set: [(lc index, point index)]; points: (n_points, 4) Montgomery
        limbs in point-label order.  Returns [(w affine limbs, random_v limbs or None)] per point."""
        L = _lib.lib()
        n = len(polys)
        lq = _lib.LIMBS[self.curve_id][1]
        arrs = [np.ascontiguousarray(p[0], dtype=np.uint64) for p in polys]
        ptrs = (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrs])
        lens = (ctypes.c_size_t * n)(*[len(a) for a in arrs])
        db = (ctypes.c_int64 * n)(*[-1 if p[1] is None else p[1] for p in polys])
        hid = (ctypes.c_int * n)(*[0 if p[2] is None else 1 for p in polys])
        rands = np.ascontiguousarray(rands, dtype=np.uint64)
        shifted_rands = np.ascontiguousarray(shifted_rands, dtype=np.uint64)
        offs, lp, lcf = [0], [], []
        for terms in lcs:
            for coeff, idx in terms:
                lp.append(-1 if idx is None else idx)
                lcf.append(np.asarray(coeff, dtype=np.uint64).reshape(4))
            offs.append(len(lp))
        offs_a = (ctypes.c_size_t * len(offs))(*offs)
        lp_a = (ctypes.c_int64 * len(lp))(*lp)
        lcf_a = np.ascontiguousarray(np.stack(lcf), dtype=np.uint64)
        ql = (ctypes.c_size_t * len(query_set))(*[q[0] for q in query_set])
        qp = (ctypes.c_size_t * len(query_set))(*[q[1] for q in query_set])
        pts = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 4)
        npts = len(pts)
        w = np.zeros((npts, 2 * lq), dtype=np.uint64)
        has = (ctypes.c_int * npts)()
        rv = np.zeros((npts, 4), dtype=np.uint64)
        _lib.check(L.b2m_ck_open_combinations(ck.handle, n, ptrs, lens, db, hid, _lib.ptr(rands), _lib.ptr(shifted_rands), rands.shape[1],
                                              len(lcs), offs_a, lp_a, _lib.ptr(lcf_a), len(query_set), ql, qp, npts, _lib.ptr(pts),
                                              _lib.ptr(np.ascontiguousarray(challenge_limbs, dtype=np.uint64)), _lib.ptr(w), has, _lib.ptr(rv)))
        return [(w[i], rv[i] if has[i] else None) for i in range(npts)]

    # -- PC::commit (Level 1) ------------------------------------------------------------------------------
    def commit(self, srs, polys, zk_rng=None):
        """`PC::commit(ck, polynomials, rng)` [reference src/lib.rs:125,172,193,213].  polys: list of
        (coeff_limbs uint64[n,4] Montgomery, degree_bound or None, hiding_bound or None).
        Returns (comms, shifted_comms, rands, shifted_rands) as limb arrays; rands are 4 Fr per polynomial."""
        L = _lib.lib()
        n = len(polys)
        lq = _lib.LIMBS[self.curve_id][1]
        arrs = [np.ascontiguousarray(p[0], dtype=np.uint64) for p in polys]
        ptrs = (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrs])
        lens = (ctypes.c_size_t * n)(*[len(a) for a in arrs])
        db = (ctypes.c_int64 * n)(*[-1 if p[1] is None else p[1] for p in polys])
        hb = (ctypes.c_int64 * n)(*[-1 if p[2] is None else p[2] for p in polys])
        comm = np.zeros((n, 2 * lq), dtype=np.uint64)
        shifted = np.zeros((n, 2 * lq), dtype=np.uint64)
        rand = np.zeros((n, 4, 4), dtype=np.uint64)
        srand = np.zeros((n, 4, 4), dtype=np.uint64)
        rp = ctypes.byref(zk_rng.c) if zk_rng is not None else None
        if isinstance(srs, CommitterKey):  # `PC::commit(ck, ..)` with the committer key's degree / bound checks
            _lib.check(L.b2m_ck_commit(srs.handle, n, ptrs, lens, db, hb, rp, _lib.ptr(comm), _lib.ptr(shifted), _lib.ptr(rand), _lib.ptr(srand), 4))
        else:
            _lib.check(L.b2m_pc_commit(srs.handle, self.pc, n, ptrs, lens, db, hb, rp, _lib.ptr(comm), _lib.ptr(shifted), _lib.ptr(rand),
                                       _lib.ptr(srand), 4))
        return comm, shifted, rand, srand

    def open(self, srs, polys, rands, shifted_rands, point_limbs, challenge_limbs, max_degree_bound=None):
        """`PC::open_individual_opening_challenges` at one point [U marlin_pc / sonic_pc open].  polys as in `commit`
        (coeff limbs, degree_bound, _), rands / shifted_rands as returned by `commit`; point and opening challenge are
        Montgomery Fr limbs.  Returns (w affine limbs, random_v limbs or None)."""
        L = _lib.lib()
        n = len(polys)
        lq = _lib.LIMBS[self.curve_id][1]
        arrs = [np.ascontiguousarray(p[0], dtype=np.uint64) for p in polys]
        ptrs = (ctypes.c_void_p * n)(*[a.ctypes.data for a in arrs])
        lens = (ctypes.c_size_t * n)(*[len(a) for a in arrs])
        db = (ctypes.c_int64 * n)(*[-1 if p[1] is None else p[1] for p in polys])
        rands = np.ascontiguousarray(rands, dtype=np.uint64)
        shifted_rands = np.ascontiguousarray(shifted_rands, dtype=np.uint64)
        w = np.zeros(2 * lq, dtype=np.uint64)
        rv = np.zeros(4, dtype=np.uint64)
        has = ctypes.c_int(0)
        _lib.check(L.b2m_pc_open(srs.handle, self.pc, n, ptrs, lens, db, _lib.ptr(rands), _lib.ptr(shifted_rands), rands.shape[1],
                                 -1 if max_degree_bound is None else max_degree_bound, _lib.ptr(np.ascontiguousarray(point_limbs)),
                                 _lib.ptr(np.ascontiguousarray(challenge_limbs)), _lib.ptr(w), ctypes.byref(has), _lib.ptr(rv)))
        return w, (rv if has.value else None)

    # -- index -----------------------------------------------------------------------------------------
    def index(self, srs, r1cs):
        """[reference src/lib.rs:100-148] -> IndexProverKey (device resident); .vk_bytes is `index_vk` (ToBytes)."""
        L = _lib.lib()
        h = ctypes.c_void_p()
        a, b, c = r1cs.matrices()
        _lib.check(L.b2m_index_create(srs.handle, self.pc, r1cs.num_constraints, r1cs.num_variables, r1cs.num_instance,
                                      ctypes.byref(a), ctypes.byref(b), ctypes.byref(c), ctypes.byref(h)))
        return IndexProverKey(srs, h, r1cs, self.pc)

    # -- prove -----------------------------------------------------------------------------------------
    def prove(self, index_pk, r1cs, zk_rng):
        """[reference src/lib.rs:151-311] -> `CanonicalSerialize` bytes of `Proof<F, PC>`.
        r1cs = None proves the instance previously copied to the GPU with `stage`."""
        L = _lib.lib()
        buf = (ctypes.c_uint8 * 2048)()
        n = ctypes.c_size_t(0)
        if r1cs is None:
            _lib.check(L.b2m_prove(index_pk.handle, None, 0, None, 0, ctypes.byref(zk_rng.c), buf, 2048, ctypes.byref(n)))
        else:
            inst = np.ascontiguousarray(r1cs.instance)
            wit = np.ascontiguousarray(r1cs.witness)
            _lib.check(L.b2m_prove(index_pk.handle, _lib.ptr(inst), len(inst), _lib.ptr(wit), len(wit), ctypes.byref(zk_rng.c), buf,
                                   2048, ctypes.byref(n)))
        return bytes(buf[:n.value])

    def stage(self, index_pk, r1cs):
        """Copy (x, w) into HBM ahead of time (device-resident timing in bench.py)."""
        inst = np.ascontiguousarray(r1cs.instance)
        wit = np.ascontiguousarray(r1cs.witness)
        _lib.check(_lib.lib().b2m_index_stage(index_pk.handle, _lib.ptr(inst), len(inst), _lib.ptr(wit), len(wit)))

    # -- verify ----------------------------------------------------------------------------------------
    def _verifier(self, vk_bytes, max_degree_, g, gamma_g, h, beta_h, bounds, bound_points):
        L = _lib.lib()
        out = ctypes.c_void_p()
        b = np.asarray(bounds, dtype=np.uint64)
        pts = np.frombuffer(b"".join(bound_points), dtype=np.uint8)
        buf = lambda x: np.frombuffer(bytes(x), dtype=np.uint8)  # noqa: E731
        vk, g_, gg, h_, bh = buf(vk_bytes), buf(g), buf(gamma_g), buf(h), buf(beta_h)
        _lib.check(L.b2m_verifier_create(self.ctx.handle, self.curve_id, self.pc, _lib.ptr(vk), len(vk), _lib.ptr(g_), _lib.ptr(gg), _lib.ptr(h_),
                                         _lib.ptr(bh), max_degree_, len(b), _lib.ptr(b) if len(b) else None, _lib.ptr(pts) if len(pts) else None,
                                         ctypes.byref(out)))
        return VerifierKey(self.ctx, self.curve_id, self.pc, out, bytes(vk_bytes))

    def verifier_key(self, pk):
        """The verifier key of an index made by `index` (reference `IndexVerifierKey` + the trimmed PC verifier key).  The G2 half
        comes from the SRS's trapdoor (a test SRS) or from the file it was loaded from, as in `UniversalSRS.save`."""
        from . import srsfile
        srs = pk.srs
        L = _lib.lib()
        cid = self.curve_id
        md = srs.max_degree
        bounds = _index_bounds(pk.vk_bytes)
        g1 = 2 * srsfile.fq_bytes(cid)

        def g1_bytes(limbs):
            limbs = np.ascontiguousarray(np.asarray(limbs, dtype=np.uint64).reshape(-1, 2 * _lib.LIMBS[cid][1]))
            out = np.zeros(len(limbs) * g1, dtype=np.uint8)
            _lib.check(L.b2m_g1_to_uncompressed(self.ctx.handle, cid, _lib.ptr(limbs), len(limbs), _lib.ptr(out)))
            return out.tobytes()

        if srs.trapdoor is not None:
            h, beta_h, neg = srsfile.g2_setup(cid, fields.FR_MODULUS[cid], srs.trapdoor[0], md, bounds)
        elif srs.g2 is not None:
            h, beta_h, neg = srs.g2
        else:
            raise ValueError("this SRS has no G2 half (neither a trapdoor nor a source file)")
        g = g1_bytes(srs.powers_limbs[0])
        gamma_g = g1_bytes(srs.gamma_limbs[list(srs.gamma_indices).index(0)])
        if self.pc == _lib.PC_MARLIN_KZG10:
            points = [g1_bytes(srs.powers_limbs[md - d]) for d in bounds]
        else:
            points = [neg[md - d] for d in bounds]
        return self._verifier(pk.vk_bytes, md, g, gamma_g, h, beta_h, bounds, points)

    def verifier_key_from_files(self, srs_path, index_vk_tobytes):
        """The verifier key from public data only: an SRS file (marlin_b200/srsfile.py layout) and the index_vk ToBytes image."""
        from . import srsfile
        d = srsfile.read_srs(srs_path)
        if d["curve_id"] != self.curve_id:
            raise ValueError(f"{srs_path} holds curve {d['curve_id']}, this Marlin instance is curve {self.curve_id}")
        g1 = 2 * srsfile.fq_bytes(self.curve_id)
        md = len(d["powers"]) // g1 - 1
        bounds = _index_bounds(index_vk_tobytes)
        if self.pc == _lib.PC_MARLIN_KZG10:
            points = [d["powers"][(md - b) * g1:(md - b + 1) * g1] for b in bounds]
        else:
            missing = [b for b in bounds if md - b not in d["neg_powers"]]
            if missing:
                raise ValueError(f"{srs_path} holds no beta^-(D - d) h for the degree bounds {missing}")
            points = [d["neg_powers"][md - b] for b in bounds]
        return self._verifier(bytes(index_vk_tobytes), md, d["powers"][:g1], d["gamma"][0], d["h"], d["beta_h"], bounds, points)

    def batch_verify(self, vk, items, rng=None):
        """`Marlin::verify` [reference src/lib.rs:315-433] for [(public_input, proof_bytes), ...] of one index -> [bool].  The public
        input is canonical ints without the leading one (`R1CS.public_input()`).  rng: the randomisers of the batched pairing check
        (ZkRng / CallbackRng); None draws a fresh ChaCha stream seeded from os.urandom."""
        L = _lib.lib()
        n = len(items)
        if n == 0:
            return []
        rng = rng or ZkRng()
        r = fields.FR_MODULUS[self.curve_id]
        ins, proofs = [], []
        for pi, proof in items:
            vals = [int(v) for v in pi]
            if any(v < 0 or v >= r for v in vals):
                raise ValueError("public input element out of range")
            ins.append(_lib.ints_to_limbs([fields.fr_to_mont(self.curve_id, v) for v in vals], 4) if vals else np.zeros((0, 4), dtype=np.uint64))
            proofs.append(np.frombuffer(bytes(proof), dtype=np.uint8) if len(proof) else np.zeros(1, dtype=np.uint8))
        in_ptrs = (ctypes.c_void_p * n)(*[a.ctypes.data if len(a) else None for a in ins])
        n_in = (ctypes.c_size_t * n)(*[len(a) for a in ins])
        pr_ptrs = (ctypes.c_void_p * n)(*[a.ctypes.data for a in proofs])
        pr_len = (ctypes.c_size_t * n)(*[len(p) for _, p in items])
        verdicts = (ctypes.c_int * n)()
        _lib.check(L.b2m_verify(vk.handle, n, in_ptrs, n_in, pr_ptrs, pr_len, ctypes.byref(rng.c), verdicts))
        self.last_verdicts = [int(v) for v in verdicts]
        return [v == _lib.VERDICT_ACCEPT for v in self.last_verdicts]

    def verify(self, vk, public_input, proof, rng=None):
        """`Marlin::verify` for one proof -> bool."""
        return self.batch_verify(vk, [(public_input, proof)], rng)[0]
