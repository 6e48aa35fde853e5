"""GPU tests at sizes the oracle cannot reach in seconds, through size-independent properties of the path
(BASELINE.json configs): contribute is a group action, so contributing (tau, alpha, beta) and then their
inverses must give back the original accumulator byte for byte; a verified response must satisfy
sx = tau * s for every vector, and its (s, sx) are the exact sums of the known discrete logs whether the round is
verified whole or shard by shard; decompress(compress(x)) = x; phase-2 batch_mul by delta then delta^-1 is the
identity.  Sizes: 2^18 powers by default; SS_TEST_FULL=1 runs BASELINE.json's own sizes — 2^22 BLS12-377 (configs[3], the
metric's configuration) and 2^21 BW6-761 (configs[2]); logs under profiles/."""
import hashlib
import os
import random

import pytest

import coracle as O
import pyref as R
import pyref_host as H
import snark_setup_b200 as S

pytestmark = pytest.mark.gpu
FULL = os.environ.get("SS_TEST_FULL") == "1"


def _scalar(label, r):
    return int.from_bytes(hashlib.blake2b(label, digest_size=64).digest(), "little") % (r - 2) + 2


def _blank(cv, rp):
    """All-generators accumulator built with bytes arithmetic (fast)."""
    out = bytearray(rp.get_length(False))
    for vec, (o, c, s) in enumerate(rp.split_offsets(False)):
        g = cv.g2 if vec in (1, 4) else cv.g1
        out[o:o + c * s] = g.encode(g.gen, False) * c
    return bytes(out)


@pytest.mark.parametrize("curve,power", [("bls12_377", 22 if FULL else 18), ("bw6_761", 21 if FULL else 12)])
def test_contribute_inverse_roundtrip_and_verify(curve, power):
    cv = R.CURVES[curve]
    cid = S.BLS12_377 if curve == "bls12_377" else S.BW6_761
    rp = R.Phase1Parameters(cv, power, 256)
    sp = S.Phase1Parameters(cid, power, 256)
    k0 = [_scalar(b"prop-0-%d" % i, cv.r) for i in range(3)]
    k1 = [_scalar(b"prop-1-%d" % i, cv.r) for i in range(3)]
    k1inv = [pow(x, -1, cv.r) for x in k1]
    chal = bytearray(sp.get_length(False))
    S.phase1_computation(sp, _blank(cv, rp), chal, False, False, S.CHECK_NO, *k0)
    chal = bytes(chal)
    resp = bytearray(sp.get_length(True))
    S.phase1_computation(sp, chal, resp, False, True, S.CHECK_NO, *k1)
    # spot parity against the oracle at a few places of every vector
    for vec, ((o, c, s), (oo, _, so)) in enumerate(zip(rp.split_offsets(False), rp.split_offsets(True))):
        grp = 1 if vec in (1, 4) else 0
        coeff = [None, None, k1[1], k1[2], k1[2]][vec]
        for i0 in sorted({0, c // 3, max(0, c - 3)}):
            n = min(3, c - i0)
            tau = 1 if vec == 4 else k1[0]
            want = O.apply_powers(cid, grp, chal[o + i0 * s:o + (i0 + n) * s], False, 3, True, n, tau=tau, first_power=i0, coeff=coeff)
            assert bytes(resp[oo + i0 * so:oo + (i0 + n) * so]) == want, (vec, i0)
    # verification of the response: new challenge + ratio pairs
    newc = bytearray(sp.get_length(False))
    seed = hashlib.blake2b(b"rho", digest_size=32).digest()
    pairs = S.phase1_verification_vectors(sp, bytes(resp), True, newc, False, seed=seed)
    tau_acc = k0[0] * k1[0] % cv.r
    for (s_, sx), grp in zip(pairs, (0, 1, 0, 0)):
        assert O.apply_powers(cid, grp, s_, False, 3, False, 1, powers=[tau_acc]) == sx
    # the exact pairs: element i of a vector is coef * t^i * G and rho_i is keyed by the vector-relative index, so
    # (s, sx) = coef * (sum_i rho_i t^i) * (G, t * G) over the n - 1 pairs
    coefs = (1, 1, k0[1] * k1[1], k0[2] * k1[2])
    for vec, ((s_, sx), coef) in enumerate(zip(pairs, coefs)):
        g = cv.g2 if vec == 1 else cv.g1
        rho = H.rho(seed, 0, rp.split_offsets(True)[vec][1] - 1)
        acc, t_i = 0, 1
        for x in rho:
            acc += x * t_i
            t_i = t_i * tau_acc % cv.r
        k = coef * acc % cv.r
        assert (s_, sx) == (g.encode(g.mul(g.gen, k), False), g.encode(g.mul(g.gen, k * tau_acc % cv.r), False)), vec
    # the same round verified shard by shard: the partial pairs add up to the same bytes
    for world in ((4, 8) if FULL else (3, 8)):
        blobs = [S.phase1_verification_vectors(sp, bytes(resp), True, None, False, seed=seed, shard=(r, world), raw=True)
                 for r in range(world)]
        assert S.phase1_reduce_partial_pairs(cid, blobs) == pairs, world
    # contribute the inverse keys on the new challenge: back to the first challenge, byte for byte
    back = bytearray(sp.get_length(False))
    S.phase1_computation(sp, bytes(newc), back, False, False, S.CHECK_NO, *k1inv)
    assert bytes(back[64:]) == chal[64:]
    # decompress(response) == new challenge (accumulator.rs:352-388 round trip)
    assert S.phase1_decompress(sp, bytes(resp))[64:] == bytes(newc[64:])
    # a single flipped byte in tau_g1 is caught: either undecodable / out of subgroup, or the ratio breaks
    o, c, s = rp.split_offsets(True)[0]
    bad = bytearray(resp)
    bad[o + 12345 % c * s + 7] ^= 0x10
    try:
        p2 = S.phase1_verification_vectors(sp, bytes(bad), True, None, False, seed=bytes(32))
        s_, sx = p2[0]
        assert O.apply_powers(cid, 0, s_, False, 3, False, 1, powers=[tau_acc]) != sx
    except (S.InvalidData, S.IncorrectSubgroup, S.PointAtInfinity):
        pass


def test_phase2_batch_mul_roundtrip_and_ratio():
    """phase2/src/parameters.rs:286-307,393-407: H <- delta^-1 H; verify via merge_pairs(before, after)."""
    cv, cid, g = R.BLS12_377, S.BLS12_377, R.BLS12_377.g1
    n = (1 << (20 if FULL else 17)) - 1  # |H| = 2^k - 1
    gen = g.encode(g.gen, False) * n
    before = S.apply_powers(cid, S.G1, gen, False, S.CHECK_NO, False, n, tau=_scalar(b"p2", cv.r), first_power=1)
    delta = _scalar(b"delta", cv.r)
    dinv = pow(delta, -1, cv.r)
    after = bytearray(before)
    S.batch_mul(cid, S.G1, after, dinv)
    assert bytes(after[:96 * 4]) == O.apply_powers(0, 0, before[:96 * 4], False, 3, False, 4, powers=[dinv] * 4)
    s, sx = S.merge_pairs(cid, S.G1, before, bytes(after), False, seed=bytes(range(32)))
    assert O.apply_powers(0, 0, s, False, 3, False, 1, powers=[dinv]) == sx
    S.check_subgroup(cid, S.G1, bytes(after), False)
    back = bytearray(after)
    S.batch_mul(cid, S.G1, back, delta)
    assert bytes(back) == before
