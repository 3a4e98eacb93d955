"""Batches of several MSM jobs through `b2m_pc_commit` (MarlinKZG10): the bucket passes of one batch alternate between two
streams and share sort slots and per-stream scratch (csrc/msm_impl.cuh run_batch), so every commitment of a batch must
equal the oracle's `PC::commit` and the same polynomial committed on its own.  The batches mix lengths (one polynomial
much longer than the rest, so the two streams are unbalanced), an all-zero and an empty polynomial, hiding polynomials
(blinding scalars in the same job) and degree-bounded ones (a commitment and its shifted commitment read the same
scalars inside one batch).  Each batch runs with the default settings and with the batched-affine levels forced on at
these small sizes."""
import random

import pytest

import b2m_testutil as util
from marlin_b200 import api
from oracle import ec, kzg
from oracle import rng as orng
from oracle.params import BLS12_381, BN254

pytestmark = pytest.mark.gpu

D = 511  # SRS degree: the long polynomial fills it, the others are 10-60 coefficients
BOUNDS = [40, 200]
SEED = bytes(range(32))


def batch_polys(curve, jobs, rnd):
    """(label, coefficients, degree_bound, hiding_bound) with exactly `jobs` MSM jobs under MarlinKZG10 (a bounded
    polynomial is two jobs: the commitment and the shifted commitment)."""
    f = curve.fr
    rv = lambda k: [rnd.randrange(f.p) for _ in range(k)]  # noqa: E731
    long_ = ("long", rv(D + 1), None, None)
    zero = ("zero", [0] * 37, None, 1)
    if jobs == 2:
        return [long_, zero]
    if jobs == 5:
        return [("b40", rv(41), 40, None), long_, zero, ("short", rv(13), None, 1)]
    assert jobs == 8
    return [("b40h", rv(30), 40, 1), long_, ("b200", rv(201), 200, None), ("empty", [], None, None), zero, ("mid", rv(60), None, 1)]


@pytest.fixture(scope="module", params=[BLS12_381, BN254], ids=lambda c: c.name)
def setup(request):
    curve = request.param
    osrs = kzg.UniversalParams(curve, D, 0x5eed1234 + len(curve.name), ec.scalar_mul(curve, 3, curve.g), 11)
    ck = kzg.CommitterKey(osrs, D, 1, BOUNDS, kzg.MARLIN)
    expected = {}
    for jobs in (2, 5, 8):
        polys = batch_polys(curve, jobs, random.Random(100 + jobs))
        ocomms, _ = kzg.commit(kzg.Engine(False), ck, [kzg.LabeledPoly(*p) for p in polys], orng.ChaChaRng(SEED, 12))
        expected[jobs] = (polys, ocomms)
    return curve, osrs, expected


@pytest.mark.parametrize("forced", [False, True], ids=["default", "levels_forced"])
@pytest.mark.parametrize("jobs", [2, 5, 8])
def test_commit_batch(b2m_ctx, monkeypatch, setup, jobs, forced):
    curve, osrs, expected = setup
    if forced:
        monkeypatch.setenv("B2M_MSM_AFFINE_MIN_REFS", "0")  # read when the SRS (and its MSM engine) is created
    polys, ocomms = expected[jobs]
    ctx = api.Context.__new__(api.Context)
    ctx.handle = b2m_ctx
    m = api.Marlin(curve.name, "marlin_kzg10", ctx=ctx)
    srs = m.srs_from_points(util.points_to_limbs(curve, osrs.powers_of_g),
                            util.points_to_limbs(curve, [osrs.power_of_gamma_g(i) for i in (0, 1, 2)]), [0, 1, 2])
    try:
        args = [(util.fr_to_mont_limbs(curve, c), d, h) for _, c, d, h in polys]
        comm, shifted, _, _ = m.commit(srs, args, api.ZkRng(SEED, 12))
        got = util.points_from_limbs(curve, comm)
        got_shifted = util.points_from_limbs(curve, shifted)
        assert got == [c.comm for c in ocomms]
        for i, (_, _, d, _) in enumerate(polys):
            if d is not None:
                assert got_shifted[i] == ocomms[i].shifted
        # one polynomial per call: draws from a continued stream reproduce the batch's blinding values
        grng = api.ZkRng(SEED, 12)
        for i, a in enumerate(args):
            c1, s1, _, _ = m.commit(srs, [a], grng)
            assert util.points_from_limbs(curve, c1)[0] == got[i]
            if a[1] is not None:
                assert util.points_from_limbs(curve, s1)[0] == got_shifted[i]
    finally:
        srs.close()
