"""Index-range shards of ONE ceremony through the C ABI (SURVEY.md §8e) — the path bench.py runs with one process per
GPU, exercised here on ONE device by calling every shard in turn: the assembled response / new challenge must be the
bytes of the unsharded call (and of the oracle), the reduced partial (s, sx) the pairs of the unsharded call, and the
four ratio verdicts those of the reference (phase1/src/computation.rs:16-193, verification.rs:217-411,
setup-utils/src/helpers.rs:371-390,406-424).  Also: Groth16 CHUNKED verification with the ratio check
(verification.rs:229-300), Marlin initialization, the strict-unchecked-inputs switch and the off-curve subgroup verdict."""
import random

import pytest

import coracle as O
import pyref as R
import snark_setup_b200 as S
from snark_setup_b200 import sharding

pytestmark = pytest.mark.gpu


def _ceremony(power, batch, seed):
    cv = R.BLS12_377
    rng = random.Random(seed)
    rp = R.Phase1Parameters(cv, power, batch)
    sp = S.Phase1Parameters(S.BLS12_377, power, batch)
    k0 = [rng.randrange(2, cv.r) for _ in range(3)]
    k1 = [rng.randrange(2, cv.r) for _ in range(3)]
    args = (rp.g1_chunk_size, rp.other_chunk_size, 0)
    chal = O.phase1_computation(0, bytes(R.phase1_initialization(rp, False)), rp.get_length(False), False, False, 3, *args, *k0)
    return cv, rp, sp, k0, k1, args, chal


@pytest.mark.parametrize("power,world", [(5, 1), (5, 2), (5, 3), (6, 8), (2, 8), (1, 4), (10, 8), (12, 3)])
def test_sharded_round_equals_whole(power, world):
    """contribute + verify, shard by shard into the same buffers; world > elements leaves empty shards (identity partials).
    From 2^10 powers on, a shard's vectors are short enough to pick a narrower MSM window than the whole vector."""
    cv, rp, sp, k0, k1, args, chal = _ceremony(power, 8, 100 + power * 10 + world)
    want = O.phase1_computation(0, chal, rp.get_length(True), False, True, 3, *args, *k1)
    resp = bytearray(sp.get_length(True))
    for r in range(world):
        S.phase1_computation(sp, chal, resp, False, True, S.CHECK_NO, *k1, shard=(r, world))
    assert bytes(resp[64:]) == want[64:]
    # verification: every shard reads the response (one overlap element) and writes its part of the new challenge
    seed = bytes(range(32))
    newc = bytearray(sp.get_length(False))
    blobs = [S.phase1_verification_vectors(sp, bytes(resp), True, newc, False, seed=seed, shard=(r, world), raw=True)
             for r in range(world)]
    full = O.phase1_computation(0, chal, rp.get_length(False), False, False, 3, *args, *k1)
    assert bytes(newc[64:]) == full[64:]
    whole = S.phase1_verification_vectors(sp, bytes(resp), True, None, False, seed=seed, raw=True)
    # rho_i is keyed by the global element index, so the sum of the partials IS the whole-vector pair
    assert S.phase1_reduce_partial_pairs(S.BLS12_377, blobs, raw=True) == whole
    tau = k0[0] * k1[0] % cv.r
    for (s, sx), g in zip(S.phase1_reduce_partial_pairs(S.BLS12_377, blobs), (cv.g1, cv.g2, cv.g1, cv.g1)):
        assert g.mul(g.decode(s, False), tau) == g.decode(sx, False)
    # the four verdicts from the reduced blob
    offs = rp.split_offsets(False)
    g1_check = bytes(newc[offs[0][0]:offs[0][0] + 2 * 96])
    g2_check = bytes(newc[offs[1][0]:offs[1][0] + 2 * 192])
    S.phase1_check_ratio_pairs(S.BLS12_377, S.phase1_reduce_partial_pairs(S.BLS12_377, blobs, raw=True), g1_check, g2_check)


def test_sharded_verdict_finds_the_tampered_vector():
    """a bad element whose ratio pair straddles two shards: the reduced verdict names the vector; an off-subgroup /
    infinity element is reported by the shard that owns it with the vector-relative index."""
    cv, rp, sp, k0, k1, args, chal = _ceremony(5, 8, 4242)
    resp = bytearray(O.phase1_computation(0, chal, rp.get_length(True), False, True, 3, *args, *k1))
    world = 4
    offs = rp.split_offsets(True)
    o, c, sz = offs[2]  # alpha_g1
    s1, e1 = sharding.shard_range(c, 1, world)
    bad = bytearray(resp)
    bad[o + e1 * sz:o + (e1 + 1) * sz] = cv.g1.encode(cv.g1.mul(cv.g1.gen, 12345), True)  # first element of shard 2
    blobs = [S.phase1_verification_vectors(sp, bytes(bad), True, None, False, seed=bytes(32), shard=(r, world), raw=True)
             for r in range(world)]
    newc = S.phase1_decompress(sp, bytes(resp))
    ou = rp.split_offsets(False)
    g1_check, g2_check = newc[ou[0][0]:ou[0][0] + 192], newc[ou[1][0]:ou[1][0] + 384]
    with pytest.raises(S.InvalidRatio) as ei:
        S.phase1_check_ratio_pairs(S.BLS12_377, S.phase1_reduce_partial_pairs(S.BLS12_377, blobs, raw=True), g1_check, g2_check)
    assert ei.value.index == 2
    # infinity in beta_g1, owned by shard 3
    o, c, sz = offs[3]
    inf = bytearray(resp)
    idx = c - 2
    inf[o + idx * sz:o + (idx + 1) * sz] = cv.g1.encode(None, True)
    for r in range(world):
        s0, e0 = sharding.shard_range(c, r, world)
        if s0 <= idx < e0 or (idx == e0 and e0 < c):  # owner, or the previous shard reading it as its overlap element
            with pytest.raises(S.PointAtInfinity) as ei:
                S.phase1_verification_vectors(sp, bytes(inf), True, None, False, seed=bytes(32), shard=(r, world))
            assert ei.value.index == idx
        else:
            S.phase1_verification_vectors(sp, bytes(inf), True, None, False, seed=bytes(32), shard=(r, world))


def test_sharded_round_device_buffers():
    """the *_shard_dev twins bench.py times: device-resident buffers, same bytes."""
    import torch
    cv, rp, sp, k0, k1, args, chal = _ceremony(6, 16, 777)
    dev = torch.device("cuda", 0)
    d_in = torch.frombuffer(bytearray(chal), dtype=torch.uint8).to(dev)
    d_out = torch.zeros(sp.get_length(True), dtype=torch.uint8, device=dev)
    d_nc = torch.zeros(sp.get_length(False), dtype=torch.uint8, device=dev)
    world = 3
    for r in range(world):
        S.phase1_computation_dev(sp, d_in.data_ptr(), d_in.numel(), d_out.data_ptr(), d_out.numel(), False, True, S.CHECK_NO,
                                 *k1, shard=(r, world))
    want = O.phase1_computation(0, chal, rp.get_length(True), False, True, 3, *args, *k1)
    assert d_out.cpu().numpy().tobytes()[64:] == want[64:]
    blobs = [S.phase1_verification_vectors_dev(sp, d_out.data_ptr(), d_out.numel(), True, d_nc.data_ptr(), d_nc.numel(), False,
                                               seed=bytes(32), shard=(r, world), raw=True) for r in range(world)]
    full = O.phase1_computation(0, chal, rp.get_length(False), False, False, 3, *args, *k1)
    assert d_nc.cpu().numpy().tobytes()[64:] == full[64:]
    tau = k0[0] * k1[0] % cv.r
    for (s, sx), g in zip(S.phase1_reduce_partial_pairs(S.BLS12_377, blobs), (cv.g1, cv.g2, cv.g1, cv.g1)):
        assert g.mul(g.decode(s, False), tau) == g.decode(sx, False)


@pytest.mark.parametrize("chunk_index", [0, 1, 2, 3])
def test_groth16_chunked_verification_with_ratio_check(chunk_index):
    """ContributionMode::Chunked verification WITH the ratio check (verification.rs:229-300): chunk c of size 8 of a
    2^4-power ceremony — chunks 0, 1 hold all five vectors' ranges, chunks 2, 3 (>= 2^k) tau_g1 only; the (s, sx) of
    every vector present must satisfy sx = tau * s and the re-emitted chunk is the decompressed chunk."""
    cv, cid = R.BLS12_377, S.BLS12_377
    power, batch, csz = 4, 5, 8
    rng = random.Random(60 + chunk_index)
    rp = R.Phase1Parameters(cv, power, batch, R.CHUNKED_MODE, chunk_index, csz)
    sp = S.Phase1Parameters(cid, power, batch, 1, chunk_index, csz)
    t0, a0, b0 = (rng.randrange(2, cv.r) for _ in range(3))
    # a chunk of a real accumulator: element j of the chunk = tau0^(c*8 + j) * G (alpha / beta on their vectors)
    first = chunk_index * csz
    acc = bytearray(rp.get_length(False))
    for vec, (o, c, s) in enumerate(rp.split_offsets(False)):
        g = cv.g2 if vec in (1, 4) else cv.g1
        co = (1, 1, a0, b0, b0)[vec]
        pts = [g.mul(g.gen, pow(t0, first + j, cv.r) * co % cv.r) for j in range(c)] if vec != 4 else [g.mul(g.gen, b0)]
        acc[o:o + c * s] = g.write_batch(pts, False)
    tau, alpha, beta = (rng.randrange(2, cv.r) for _ in range(3))
    resp = bytearray(sp.get_length(True))
    S.phase1_computation(sp, bytes(acc), resp, False, True, S.CHECK_NO, tau, alpha, beta)
    assert bytes(resp) == bytes(R.phase1_computation(rp, bytes(acc), False, True, R.NO, tau, alpha, beta))
    newc = bytearray(sp.get_length(False))
    pairs = S.phase1_verification_vectors(sp, bytes(resp), True, newc, False, ratio_check=True, seed=bytes(range(32)))
    assert bytes(newc[64:]) == bytes(R.phase1_computation(rp, bytes(acc), False, False, R.NO, tau, alpha, beta))[64:]
    t = t0 * tau % cv.r
    present = (True, rp.other_chunk_size > 0, rp.other_chunk_size > 0, rp.other_chunk_size > 0)
    for (s, sx), g, here in zip(pairs, (cv.g1, cv.g2, cv.g1, cv.g1), present):
        if here:
            sp_ = g.decode(s, False)
            assert sp_ is not None and g.mul(sp_, t) == g.decode(sx, False)
        else:  # vector absent from this chunk: identity pair
            assert g.decode(s, False) is None and g.decode(sx, False) is None
    # a swapped pair inside the chunk breaks exactly that vector's ratio
    o, c, sz = rp.split_offsets(True)[0]
    bad = bytearray(resp)
    bad[o + 2 * sz:o + 3 * sz], bad[o + 3 * sz:o + 4 * sz] = resp[o + 3 * sz:o + 4 * sz], resp[o + 2 * sz:o + 3 * sz]
    pairs = S.phase1_verification_vectors(sp, bytes(bad), True, None, False, ratio_check=True, seed=bytes(range(32)))
    s, sx = pairs[0]
    assert cv.g1.mul(cv.g1.decode(s, False), t) != cv.g1.decode(sx, False)


@pytest.mark.parametrize("mode,chunk_index,chunk_size", [(0, 0, 0), (1, 0, 4), (1, 1, 4)])
def test_marlin_initialization_and_shards(mode, chunk_index, chunk_size):
    """ProvingSystem::Marlin: initialization fills tau_g1 and, on chunk 0, the k+2 tau_g2 and 3+3k alpha_g1 generators —
    no beta slots (buffers.rs:246-288, initialization.rs:12-57); sharded computation == whole computation."""
    cv, cid = R.BLS12_377, S.BLS12_377
    power, batch = 3, 8
    rp = R.Phase1Parameters(cv, power, batch, mode, chunk_index, chunk_size, R.MARLIN)
    sp = S.Phase1Parameters(cid, power, batch, mode, chunk_index, chunk_size, 1)
    for compressed in (False, True):
        assert S.phase1_initialization(sp, compressed) == bytes(R.phase1_initialization(rp, compressed))
    rng = random.Random(31 + chunk_index)
    tau, alpha = rng.randrange(2, cv.r), rng.randrange(2, cv.r)
    acc = S.phase1_initialization(sp, False)
    want = bytes(R.phase1_computation(rp, acc, False, True, R.NO, tau, alpha, 0))
    out = bytearray(sp.get_length(True))
    for r in range(3):
        S.phase1_computation(sp, acc, out, False, True, S.CHECK_NO, tau, alpha, 1, shard=(r, 3))
    assert bytes(out) == want


def _off_subgroup_point(g, rng):
    """a curve point outside the order-r subgroup"""
    F = g.F
    while True:
        x = rng.randrange(F.p) if F.degree == 1 else (rng.randrange(F.p), rng.randrange(F.p))
        y = F.sqrt(F.add(F.mul(F.sqr(x), x), g.b))
        if y is not None and not g.in_subgroup((x, y)):
            return (x, y)


@pytest.mark.parametrize("gname", ["g1", "g2"])
def test_strict_unchecked_inputs_matches_mul_bigint_off_subgroup(gname):
    """CheckForCorrectness::No lets any point through; with ss_set_strict_unchecked_inputs(1) the product of an
    OFF-SUBGROUP base is what ark-ec's mul_bigint gives (the oracle's double-and-add), which GLV / GLS would not."""
    cv, cid = R.BLS12_377, S.BLS12_377
    g, gid = (cv.g1, S.G1) if gname == "g1" else (cv.g2, S.G2)
    rng = random.Random(99)
    pts = [_off_subgroup_point(g, rng) for _ in range(3)] + [g.mul(g.gen, 7)]
    ks = [rng.randrange(cv.r) for _ in pts]
    buf = g.write_batch(pts, False)
    want = O.apply_powers(0, gid, buf, False, 3, True, len(pts), powers=ks)
    assert want == g.write_batch([g.mul(P, k) for P, k in zip(pts, ks)], True)
    try:
        S.set_strict_unchecked_inputs(True)
        got = S.apply_powers(cid, gid, buf, False, S.CHECK_NO, True, len(pts), powers=ks)
    finally:
        S.set_strict_unchecked_inputs(False)
    assert got == want
    # the default path agrees on the subgroup element (and is allowed to differ on the others)
    fast = S.apply_powers(cid, gid, buf, False, S.CHECK_NO, True, len(pts), powers=ks)
    sz = g.size(True)
    assert fast[3 * sz:] == want[3 * sz:]


@pytest.mark.parametrize("gname", ["g1", "g2"])
def test_subgroup_verdict_on_off_curve_uncompressed_input(gname):
    """check_subgroup on UNCOMPRESSED elements read without validation: an off-curve element gets the verdict of the
    reference's r*P on its own formulas (accumulator.rs:120-137), i.e. the oracle's."""
    cv, cid = R.BLS12_377, S.BLS12_377
    g, gid = (cv.g1, S.G1) if gname == "g1" else (cv.g2, S.G2)
    rng = random.Random(5)
    good = [g.mul(g.gen, rng.randrange(1, cv.r)) for _ in range(6)]
    buf = bytearray(g.write_batch(good, False))
    S.check_subgroup(cid, gid, bytes(buf), False)
    # off-curve: bump y of element 4 (stays a canonical field element)
    sz = g.size(False)
    x, y = good[4]
    y2 = g.F.add(y, g.F.from_int(1))
    buf[4 * sz:5 * sz] = g.encode((x, y2), False)
    try:
        O.transcode(0, gid, bytes(buf), False, 3, False, 6, rmul_subgroup=True, want_output=False)
        oracle_ok = True
    except O.OracleError as e:
        oracle_ok = False
        assert e.index == 4
    if oracle_ok:
        S.check_subgroup(cid, gid, bytes(buf), False)
    else:
        with pytest.raises(S.IncorrectSubgroup) as ei:
            S.check_subgroup(cid, gid, bytes(buf), False)
        assert ei.value.index == 4


def test_beta_g2_is_validated_without_a_new_challenge():
    """verification.rs:199-201 reads beta_g2 with check_output_for_correctness whatever happens to the new challenge:
    an infinite or off-subgroup beta_g2 is rejected by the aggregate-style call (new_challenge = None) too."""
    cv, rp, sp, k0, k1, args, chal = _ceremony(3, 8, 31337)
    resp = bytearray(O.phase1_computation(0, chal, rp.get_length(True), False, True, 3, *args, *k1))
    S.phase1_verification_vectors(sp, bytes(resp), True, None, False, seed=bytes(32))
    o, c, sz = rp.split_offsets(True)[4]
    bad = bytearray(resp)
    bad[o:o + sz] = cv.g2.encode(None, True)
    with pytest.raises(S.PointAtInfinity):
        S.phase1_verification_vectors(sp, bytes(bad), True, None, False, seed=bytes(32))
    rng = random.Random(3)
    bad[o:o + sz] = cv.g2.encode(_off_subgroup_point(cv.g2, rng), True)
    with pytest.raises(S.InvalidData):  # Validate::Yes fails (arkworks reports InvalidData for a point outside the subgroup)
        S.phase1_verification_vectors(sp, bytes(bad), True, None, False, seed=bytes(32))
