"""How the host driver fans a phase-1 call out over vectors (and shards), with the vectors running concurrently and one
after another: a failing element is reported with its vector-relative index and its vector's name, the lowest-numbered
failing vector wins when several fail, and Marlin contribute gives the reference's bytes whichever way it is scheduled."""
import random

import pytest

import coracle as O
import pyref as R
import snark_setup_b200 as S
from snark_setup_b200 import ffi, sharding

pytestmark = pytest.mark.gpu

POWER, BATCH, WORLD = 5, 8, 3


@pytest.fixture(params=[True, False], ids=["concurrent", "sequential"])
def concurrent(request):
    ffi.set_concurrent_vectors(request.param)
    yield request.param
    ffi.set_concurrent_vectors(True)


@pytest.fixture(scope="module")
def ceremony():
    """a compressed BLS12-377 accumulator after one contribution, and the keys of the next"""
    cv = R.BLS12_377
    rng = random.Random(2718)
    rp = R.Phase1Parameters(cv, POWER, BATCH)
    sp = S.Phase1Parameters(S.BLS12_377, POWER, BATCH)
    k0 = [rng.randrange(2, cv.r) for _ in range(3)]
    k1 = [rng.randrange(2, cv.r) for _ in range(3)]
    args = (rp.g1_chunk_size, rp.other_chunk_size, 0)
    chal = O.phase1_computation(0, bytes(R.phase1_initialization(rp, False)), rp.get_length(True), False, True, 3, *args, *k0)
    return cv, rp, sp, k1, bytes(chal)


def _tamper(cv, rp, buf, bad):
    """bad = {vector: (element index, compressed encoding)}"""
    out = bytearray(buf)
    for vec, (idx, enc) in bad.items():
        o, c, sz = rp.split_offsets(True)[vec]
        out[o + idx * sz:o + (idx + 1) * sz] = enc
    return bytes(out)


def _expect(call, shards, idx, exc, name):
    """`call(shard)` raises `exc` naming vector `name` at element `idx` in the shard that owns it; the others pass."""
    for shard, (s0, e0) in shards:
        if s0 <= idx < e0:
            with pytest.raises(exc) as ei:
                call(shard)
            assert ei.value.index == idx and name in str(ei.value), (shard, ei.value.index, str(ei.value))
        else:
            call(shard)


def _shards(c, sharded):
    if not sharded:
        return [(None, (0, c))]
    return [((r, WORLD), sharding.shard_range(c, r, WORLD)) for r in range(WORLD)]


def _undecodable(cv):
    return b"\xff" * (cv.g1.csize - 1) + b"\x3f"  # x >= p


@pytest.mark.parametrize("sharded", [False, True], ids=["whole", "shards"])
def test_computation_reports_the_failing_vector(ceremony, concurrent, sharded):
    cv, rp, sp, k1, chal = ceremony
    c = rp.other_chunk_size
    shards = _shards(c, sharded)
    idx = shards[-1][1][0] + 1  # inside the last shard, not on its boundary

    def contribute(inp):
        return lambda shard: S.phase1_computation(sp, inp, bytearray(sp.get_length(True)), True, True, S.CHECK_FULL, *k1,
                                                  shard=shard)
    _expect(contribute(_tamper(cv, rp, chal, {3: (idx, _undecodable(cv))})), shards, idx, S.InvalidData, "beta_g1")
    # alpha_g1 and beta_g1 both fail in the same shard: the lower vector is the one reported
    both = _tamper(cv, rp, chal, {2: (idx, _undecodable(cv)), 3: (idx + 1, _undecodable(cv))})
    _expect(contribute(both), shards, idx, S.InvalidData, "alpha_g1")


@pytest.mark.parametrize("sharded", [False, True], ids=["whole", "shards"])
def test_verification_reports_the_failing_vector(ceremony, concurrent, sharded):
    cv, rp, sp, k1, chal = ceremony
    c = rp.other_chunk_size
    shards = _shards(c, sharded)
    idx = shards[-1][1][0] + 1  # not the overlap element the previous shard reads for its last ratio pair
    inf = cv.g1.encode(None, True)

    def verify(resp):
        return lambda shard: S.phase1_verification_vectors(sp, resp, True, None, False, seed=bytes(32), shard=shard)
    _expect(verify(_tamper(cv, rp, chal, {3: (idx, inf)})), shards, idx, S.PointAtInfinity, "beta_g1")
    _expect(verify(_tamper(cv, rp, chal, {2: (idx, inf), 3: (idx + 1, inf)})), shards, idx, S.PointAtInfinity, "alpha_g1")


@pytest.mark.parametrize("mode,chunk_index,chunk_size", [(0, 0, 0), (1, 0, 4), (1, 1, 4)])
def test_marlin_contribute_any_schedule(concurrent, mode, chunk_index, chunk_size):
    """tau_g1 split like Groth16's powers; tau_g2 / alpha_g1 (chunk 0 only) done whole by the owner of part 0"""
    cv = R.BLS12_377
    rng = random.Random(1300 + chunk_index)
    rp = R.Phase1Parameters(cv, 3, 8, mode, chunk_index, chunk_size, R.MARLIN)
    sp = S.Phase1Parameters(S.BLS12_377, 3, 8, mode, chunk_index, chunk_size, 1)
    tau, alpha = rng.randrange(2, cv.r), rng.randrange(2, cv.r)
    acc = bytearray(rp.get_length(False))
    for vec, (o, c, s) in enumerate(rp.split_offsets(False)):
        g = cv.g2 if vec in (1, 4) else cv.g1
        acc[o:o + c * s] = g.write_batch([g.mul(g.gen, rng.randrange(1, cv.r)) for _ in range(c)], False)
    want = bytes(R.phase1_computation(rp, bytes(acc), False, True, R.NO, tau, alpha, 0))
    out = bytearray(sp.get_length(True))
    S.phase1_computation(sp, bytes(acc), out, False, True, S.CHECK_NO, tau, alpha, 1)
    assert bytes(out) == want
    out = bytearray(sp.get_length(True))
    for r in range(WORLD):
        S.phase1_computation(sp, bytes(acc), out, False, True, S.CHECK_NO, tau, alpha, 1, shard=(r, WORLD))
    assert bytes(out) == want
