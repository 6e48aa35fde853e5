"""Host-side pieces of a phase-1 round that sit AROUND the hot path (SURVEY.md §8a "host-side helpers", App. A.4):
key generation, hash_to_g2, the PublicKey record and the proof-of-knowledge checks.  TEST INFRASTRUCTURE ONLY, like
oracle/pyref.py; the Rust host keeps doing all of this itself — it is restated here so that config C1's transcript
(new -> contribute -> verify) can be produced and checked end to end without Rust.

RECALLED, UNVERIFIABLE OFFLINE.  Everything below restates third-party behaviour from memory (rand_chacha 0.3.1,
rand 0.8.5, blake2s_simd 1.0.2, blake2 0.10, ark-ff / ark-ec 0.4.2); there is no Rust toolchain here to confirm the RNG
draw order, so a byte-for-byte match of the KEYS with the reference binary is a hypothesis (the hot path does not
depend on it: keys are inputs to it).  What IS checked (tests/test_oracle_cpu.py): the construction is self-consistent —
every proof of knowledge of a generated key verifies under the oracle's pairing, and the transcript digest is pinned
so that any drift of this restatement is visible.

  derive_rng_from_seed     setup-utils/src/seed.rs:7-14        BLAKE2s-256(personal "NIM-SEED") -> ChaCha20 key
  Phase1::key_generation   phase1/src/key_generation.rs:8-53
  compute_g2_s             setup-utils/src/helpers.rs:428-443   BLAKE2b-512(personalization || digest || g1_s || g1_s_x)
  hash_to_g2               setup-utils/src/helpers.rs:277-291   ChaCha20(first 32 digest bytes) -> from_random_bytes -> cofactor
  PublicKey::write         phase1/src/objects/public_key.rs:40-55 (compressed, field-declaration order)
  PoK checks               phase1/src/verification.rs:83-133
"""
from __future__ import annotations

import hashlib

import pyref as R


# ---------------------------------------------------------------------------------------------------------------
# rand_chacha::ChaChaRng (= ChaCha20Rng): 64-bit block counter from 0, 64-bit stream id 0; the 16 output words of a
# block are consumed in order; next_u64 = two consecutive words, low first (rand_core BlockRng)
# ---------------------------------------------------------------------------------------------------------------
def _rotl(x, r):
    return ((x << r) | (x >> (32 - r))) & 0xffffffff


def _qr(s, a, b, c, d):
    s[a] = (s[a] + s[b]) & 0xffffffff; s[d] = _rotl(s[d] ^ s[a], 16)
    s[c] = (s[c] + s[d]) & 0xffffffff; s[b] = _rotl(s[b] ^ s[c], 12)
    s[a] = (s[a] + s[b]) & 0xffffffff; s[d] = _rotl(s[d] ^ s[a], 8)
    s[c] = (s[c] + s[d]) & 0xffffffff; s[b] = _rotl(s[b] ^ s[c], 7)


def chacha20_block(key: bytes, counter: int):
    k = [int.from_bytes(key[4 * i:4 * i + 4], "little") for i in range(8)]
    init = [0x61707865, 0x3320646e, 0x79622d32, 0x6b206574] + k + [counter & 0xffffffff, counter >> 32, 0, 0]
    s = list(init)
    for _ in range(10):
        _qr(s, 0, 4, 8, 12); _qr(s, 1, 5, 9, 13); _qr(s, 2, 6, 10, 14); _qr(s, 3, 7, 11, 15)
        _qr(s, 0, 5, 10, 15); _qr(s, 1, 6, 11, 12); _qr(s, 2, 7, 8, 13); _qr(s, 3, 4, 9, 14)
    return [(a + b) & 0xffffffff for a, b in zip(s, init)]


def chacha20_blocks(key: bytes, first: int, n: int):
    """chacha20_block for the counters first .. first + n - 1 at once (numpy, one lane per block) -> uint32 [n, 16].
    The pure-Python block takes minutes over the 2^21 blocks of one MSM tile."""
    import numpy as np
    k = np.frombuffer(bytes(key), dtype="<u4")
    ctr = np.arange(first, first + n, dtype=np.uint64)
    consts = (0x61707865, 0x3320646e, 0x79622d32, 0x6b206574)
    init = [np.full(n, c, np.uint32) for c in consts] + [np.full(n, w, np.uint32) for w in k]
    init += [(ctr & 0xffffffff).astype(np.uint32), (ctr >> np.uint64(32)).astype(np.uint32), np.zeros(n, np.uint32),
             np.zeros(n, np.uint32)]
    x = [v.copy() for v in init]
    t = np.empty(n, np.uint32)

    def rotl(v, r):
        np.right_shift(v, np.uint32(32 - r), out=t)
        np.left_shift(v, np.uint32(r), out=v)
        np.bitwise_or(v, t, out=v)

    def qr(a, b, c, d):
        for (p, q, s, r) in ((a, b, d, 16), (c, d, b, 12), (a, b, d, 8), (c, d, b, 7)):
            np.add(x[p], x[q], out=x[p])
            np.bitwise_xor(x[s], x[p], out=x[s])
            rotl(x[s], r)

    for _ in range(10):
        qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15)
        qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14)
    for v, v0 in zip(x, init):
        np.add(v, v0, out=v)
    return np.stack(x, axis=1)


def rho(seed: bytes, first: int, n: int):
    """The random scalars of the device ratio-check MSM (snark-setup_b200/csrc/msm.cuh): rho_i = the first 16 bytes of
    ChaCha20(key = seed, counter = first + i, nonce = 0) as a little-endian integer, for i < n."""
    raw = chacha20_blocks(seed, first, n)[:, :4].astype("<u4").tobytes()
    return [int.from_bytes(raw[16 * i:16 * i + 16], "little") for i in range(n)]


class ChaChaRng:
    def __init__(self, seed32: bytes):
        assert len(seed32) == 32
        self.key, self.ctr, self.buf = bytes(seed32), 0, []

    def next_u32(self):
        if not self.buf:
            self.buf = chacha20_block(self.key, self.ctr)
            self.ctr += 1
        return self.buf.pop(0)

    def next_u64(self):
        lo = self.next_u32()
        return lo | (self.next_u32() << 32)

    def gen_u8(self):      # Standard for u8: next_u32() as u8
        return self.next_u32() & 0xff

    def gen_bool(self):    # Standard for bool: (next_u32() as i32) < 0
        return self.next_u32() >> 31 == 1


def derive_rng_from_seed(seed: bytes) -> ChaChaRng:
    """setup-utils/src/seed.rs:7-14"""
    return ChaChaRng(hashlib.blake2s(seed, person=b"NIM-SEED").digest())


# ---------------------------------------------------------------------------------------------------------------
# ark-ff / ark-ec sampling
# ---------------------------------------------------------------------------------------------------------------
def fp_rand(p: int, rng: ChaChaRng) -> int:
    """ark-ff `Distribution<Fp> for Standard`: N random u64 limbs (limb 0 first), the bits above the modulus length
    masked off, rejected when >= p; the accepted limbs ARE the internal Montgomery representation, so the value is
    limbs * R^-1 mod p with R = 2^(64 N)."""
    n = (p.bit_length() + 63) // 64
    shave = 64 * n - p.bit_length()
    while True:
        limbs = [rng.next_u64() for _ in range(n)]
        limbs[-1] &= (1 << (64 - shave)) - 1 if shave < 64 else 0
        v = sum(l << (64 * i) for i, l in enumerate(limbs))
        if v < p:
            return v * pow(1 << (64 * n), -1, p) % p


def _point_from_x(g: R.Group, x, greatest: bool):
    """Affine::get_point_from_x_unchecked: (smaller, larger) root by the field's Ord, `greatest` picks the larger"""
    F = g.F
    y = F.sqrt(g.rhs(x))
    if y is None:
        return None
    ny = F.neg(y)
    lo, hi = (y, ny) if F.gt(ny, y) else (ny, y)
    return (x, hi if greatest else lo)


def g1_rand(cv: R.Curve, cofactor: int, rng: ChaChaRng):
    """`Distribution<Projective<P>> for Standard` (ark-ec short_weierstrass): x <- Fq::rand, greatest <- bool,
    retry until x is on the curve, then multiply by the cofactor."""
    g = cv.g1
    while True:
        x = fp_rand(g.F.p, rng)
        greatest = rng.gen_bool()
        P = _point_from_x(g, x, greatest)
        if P is not None:
            return g.mul(P, cofactor)


def _fp_from_random_bytes(p: int, b: bytes, flag_bits: int):
    """ark-ff Fp::from_random_bytes_with_flags: flags = top `flag_bits` bits of the serialized form's last byte, every bit
    above the modulus length masked away, None when the rest is >= p."""
    nbytes = (p.bit_length() + flag_bits + 7) // 8
    assert len(b) == nbytes
    flags = b[-1] & ((0xff << (8 - flag_bits)) & 0xff) if flag_bits else 0
    v = int.from_bytes(b, "little") & ((1 << p.bit_length()) - 1)
    return (v, flags) if v < p else None


def g2_from_random_bytes(g2: R.Group, b: bytes):
    """AffineRepr::from_random_bytes for a short-Weierstrass G2 over Fq2: x = (c0, c1) from the two halves (flags on the
    second), infinity only for x = 0 with the infinity flag, otherwise the root selected by the sign flag."""
    p = g2.F.p
    half = len(b) // 2
    c0 = _fp_from_random_bytes(p, b[:half], 0)
    c1 = _fp_from_random_bytes(p, b[half:], 2)
    if c0 is None or c1 is None:
        return None, False
    flags = c1[1]
    if flags == (R.FLAG_NEG | R.FLAG_INF):
        return None, False
    x = (c0[0], c1[0])
    if flags & R.FLAG_INF:
        return None, x == (0, 0)   # (identity, valid) only for x = 0; any other x with the flag is rejected
    P = _point_from_x(g2, x, bool(flags & R.FLAG_NEG))
    return P, P is not None


def hash_to_g2(cv: R.Curve, g2_cofactor: int, digest: bytes):
    """setup-utils/src/helpers.rs:277-291"""
    rng = ChaChaRng(digest[:32])
    size = cv.g2.size(True)
    while True:
        b = bytes(rng.gen_u8() for _ in range(size))
        P, ok = g2_from_random_bytes(cv.g2, b)
        if ok and P is not None:
            Q = cv.g2.mul(P, g2_cofactor)
            if Q is not None:
                return Q


def compute_g2_s(cv: R.Curve, g2_cofactor: int, digest: bytes, g1_s, g1_s_x, personalization: int):
    """setup-utils/src/helpers.rs:428-443"""
    h = hashlib.blake2b(digest_size=64)
    h.update(bytes([personalization]))
    h.update(digest)
    h.update(cv.g1.encode(g1_s, True) + cv.g1.encode(g1_s_x, True))
    return hash_to_g2(cv, g2_cofactor, h.digest())


# BLS12-377 cofactors: h1 = (u - 1)^2 / 3; h2 from the order of the sextic twist that holds G2 (found among the six
# twist orders as the one that kills a point of y^2 = x^3 + B'; computed once)
_BLS_U = 0x8508c00000000001
BLS12_377_G1_COFACTOR = (_BLS_U - 1) ** 2 // 3
_G2_COFACTOR_CACHE = {}


def bls12_377_g2_cofactor() -> int:
    if "h2" in _G2_COFACTOR_CACHE:
        return _G2_COFACTOR_CACHE["h2"]
    cv = R.BLS12_377
    q, r = R.BLS12_377_Q, cv.r
    t = q + 1 - BLS12_377_G1_COFACTOR * r
    t2 = t * t - 2 * q                       # trace over Fq2
    # 4 q^2 - t2^2 = 3 f^2
    from math import isqrt
    f = isqrt((4 * q * q - t2 * t2) // 3)
    assert 3 * f * f == 4 * q * q - t2 * t2
    g2 = cv.g2
    x = (1, 1)
    while g2.F.sqrt(g2.rhs(x)) is None:
        x = (x[0] + 1, 1)
    P = (x, g2.F.sqrt(g2.rhs(x)))
    for tt in (t2, -t2, (t2 + 3 * f) // 2, (t2 - 3 * f) // 2, (-t2 + 3 * f) // 2, (-t2 - 3 * f) // 2):
        n = q * q + 1 - tt
        if n % r == 0 and g2.mul(P, n) is None:
            _G2_COFACTOR_CACHE["h2"] = n // r
            return n // r
    raise AssertionError("no twist order found")


def key_generation(cv: R.Curve, rng: ChaChaRng, digest: bytes):
    """Phase1::key_generation (phase1/src/key_generation.rs:8-53) for BLS12-377.
    Returns (public_key dict, (tau, alpha, beta))."""
    assert len(digest) == 64 and cv is R.BLS12_377
    h1, h2 = BLS12_377_G1_COFACTOR, bls12_377_g2_cofactor()
    tau, alpha, beta = fp_rand(cv.r, rng), fp_rand(cv.r, rng), fp_rand(cv.r, rng)
    pk = {}
    for name, x, pers in (("tau", tau, 0), ("alpha", alpha, 1), ("beta", beta, 2)):
        g1_s = g1_rand(cv, h1, rng)
        g1_s_x = cv.g1.mul(g1_s, x)
        g2_s = compute_g2_s(cv, h2, digest, g1_s, g1_s_x, pers)
        pk[name + "_g1"] = (g1_s, g1_s_x)
        pk[name + "_g2"] = cv.g2.mul(g2_s, x)
    return pk, (tau, alpha, beta)


def public_key_bytes(cv: R.Curve, pk) -> bytes:
    """PublicKey::write: derive(CanonicalSerialize) in field order, compressed (public_key.rs:14-22,51)"""
    out = b""
    for name in ("tau_g1", "alpha_g1", "beta_g1"):
        out += cv.g1.encode(pk[name][0], True) + cv.g1.encode(pk[name][1], True)
    for name in ("tau_g2", "alpha_g2", "beta_g2"):
        out += cv.g2.encode(pk[name], True)
    return out


def verify_proofs_of_knowledge(cv: R.Curve, pk, digest: bytes) -> bool:
    """phase1/src/verification.rs:83-133: same_ratio((g1_s, g1_s_x), (g2_s, g2_s_x)) with g2_s re-derived from the digest"""
    h2 = bls12_377_g2_cofactor()
    for name, pers in (("tau", 0), ("alpha", 1), ("beta", 2)):
        g1_s, g1_s_x = pk[name + "_g1"]
        g2_s = compute_g2_s(cv, h2, digest, g1_s, g1_s_x, pers)
        if not R.same_ratio(cv, (g1_s, g1_s_x), (g2_s, pk[name + "_g2"])):
            return False
    return True
