"""CPU suite for prepare_phase2 on MNT4-753 / MNT6-753: the evaluation-domain constants of the two 753-bit scalar
fields (MNT4 Fr = Mnt753R, 2-adicity 30; MNT6 Fr = Mnt753Q, 2-adicity 15), the generated device header, the oracle's
two IFFT algorithms against each other on G1 and G2, and the argument checks of the C ABI that run before any device
work (non-power-of-two sizes, MNT6 domains above 2^15, non-canonical 95-byte coefficients)."""
import os
import random
import re
import sys

import pytest

import pyref as R
import snark_setup_b200 as S

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gen_constants as G  # noqa: E402

# the oracle's domains need the multiplicative generators of the MNT scalar fields (GENERATOR = 17, see
# tools/gen_constants.py); the BLS12-377 / BW6-761 entries are untouched
R.FR_GENERATOR.update(G.MNT_FFT_GENERATOR)

FIELDS = [("mnt4_753", R.MNT753_R, 30, "Mnt753R"), ("mnt6_753", R.MNT753_Q, 15, "Mnt753Q")]
CID = {"mnt4_753": S.MNT4_753, "mnt6_753": S.MNT6_753}


def _small_primes(n, limit=3000):
    return [p for p in range(2, limit) if n % p == 0 and all(p % q for q in range(2, int(p ** 0.5) + 1))]


@pytest.mark.parametrize("curve,r,s,_", FIELDS, ids=[f[0] for f in FIELDS])
def test_two_adic_root_has_exact_order(curve, r, s, _):
    assert R.curve_by_name(curve).r == r
    assert R.two_adicity(r) == s
    g = G.MNT_FFT_GENERATOR[r]
    assert g == 17 and R.FR_GENERATOR[r] == 17
    # what can be checked of the recalled generator: a quadratic non-residue (so g^t has order exactly 2^s) and no
    # l-th power for the small primes l | r - 1 (a primitive root cannot be one)
    assert pow(g, (r - 1) // 2, r) == r - 1
    assert all(pow(g, (r - 1) // l, r) != 1 for l in _small_primes(r - 1))
    w = R.get_root_of_unity(r, 1 << s)
    assert w == pow(g, (r - 1) >> s, r)
    assert pow(w, 1 << s, r) == 1 and pow(w, 1 << (s - 1), r) == r - 1
    for log_n in (0, 1, 3, s):
        wn = R.get_root_of_unity(r, 1 << log_n)
        assert pow(wn, 1 << log_n, r) == 1 and (log_n == 0 or pow(wn, 1 << (log_n - 1), r) == r - 1)
    with pytest.raises(ValueError):
        R.get_root_of_unity(r, 1 << (s + 1))


def test_generated_headers_match_the_generator():
    with open(os.path.join(ROOT, "snark-setup_b200", "csrc", "constants_gen.cuh")) as f:
        dev = f.read()
    with open(os.path.join(ROOT, "oracle", "constants_gen.h")) as f:
        orc = f.read()
    assert dev == G.emit_device()
    assert orc == G.emit_oracle()
    for _, r, s, name in FIELDS:
        body = dev[dev.index("struct %s {" % name):]
        assert re.search(r"TWO_ADICITY = (\d+);", body).group(1) == str(s)
        m = re.search(r"fft_root\(int i\) \{ const uint32_t v\[24\] = \{([^}]*)\}", body)
        limbs = [int(x.strip().rstrip("u"), 16) for x in m.group(1).split(",")]
        mont = sum(l << (32 * i) for i, l in enumerate(limbs))
        assert mont == (R.get_root_of_unity(r, 1 << s) << 768) % r


def _inputs(g, n, rng):
    """random subgroup points with identities, repeats and negations among them"""
    base = [g.mul(g.gen, rng.randrange(1, g.r)) for _ in range(max(2, n // 2))]
    pts = [rng.choice(base) for _ in range(n)]
    if n >= 4:
        pts[1] = None
        pts[2] = pts[0]
        pts[3] = g.neg(pts[0])
    return pts


@pytest.mark.parametrize("curve", ["mnt4_753", "mnt6_753"])
@pytest.mark.parametrize("grp", [0, 1])
def test_group_ifft_fast_matches_definition(curve, grp):
    cv = R.curve_by_name(curve)
    g = cv.g2 if grp else cv.g1
    rng = random.Random(31 * CID[curve] + grp)
    for n in (1, 2, 4):
        pts = _inputs(g, n, rng)
        assert R.group_ifft_fast(g, pts) == R.group_ifft(g, pts), n


@pytest.mark.parametrize("curve", ["mnt4_753", "mnt6_753"])
def test_group_ifft_of_known_discrete_logs(curve):
    """P_i = s_i G  =>  to_coeffs(P) = scalar_ifft(s) G"""
    cv = R.curve_by_name(curve)
    rng = random.Random(5 + CID[curve])
    s = [rng.randrange(cv.r) for _ in range(8)]
    s[2], s[5] = 0, s[1]
    for g in (cv.g1, cv.g2):
        pts = [g.mul(g.gen, x) for x in s]
        assert R.group_ifft_fast(g, pts) == [g.mul(g.gen, c) for c in R.scalar_ifft(cv.r, s)]


# ---- C ABI argument checks (host logic, before any device work) -------------------------------------------------
def test_domain_limits():
    c1, c2 = 95, 285
    m, b = S.groth16_params_size(S.MNT6_753, 1 << 15, True)
    assert (m, b) == (1 << 15, 2 * c1 + c2 + 3 * m * c1 + m * c2 + (m - 1) * c1)
    m, b = S.groth16_params_size(S.MNT4_753, (1 << 15) + 1, False)
    assert (m, b) == (1 << 16, 2 * 190 + 380 + 3 * m * 190 + m * 380 + (m - 1) * 190)
    assert S.groth16_params_size(S.MNT4_753, 1 << 30, True)[0] == 1 << 30
    with pytest.raises(S.InvalidArgument):  # Fr of MNT6-753 has no radix-2 domain above 2^15
        S.groth16_params_size(S.MNT6_753, (1 << 15) + 1, True)
    with pytest.raises(S.InvalidArgument):  # nor Fr of MNT4-753 above 2^30
        S.groth16_params_size(S.MNT4_753, (1 << 30) + 1, True)
    sp = S.Phase1Parameters(S.MNT6_753, 3, 8)
    with pytest.raises(S.InvalidArgument):
        S.groth16_params_new(sp, bytes(sp.get_length(False)), False, (1 << 15) + 1, False)
    with pytest.raises(S.InvalidArgument):  # group IFFT of 2^16 MNT6 points
        S.group_ifft(S.MNT6_753, S.G1, bytes(190 << 16), False, False)
    for cid, usz in ((S.MNT4_753, 190), (S.MNT6_753, 570)):
        for n in (3, 6, 12):
            with pytest.raises(S.SetupError):  # not a radix-2 domain size
                S.group_ifft(cid, S.G2 if usz == 570 else S.G1, bytes(usz * n), False, False)


@pytest.mark.parametrize("curve", ["mnt4_753", "mnt6_753"])
def test_non_canonical_coefficients_are_rejected(curve):
    cv = R.curve_by_name(curve)
    cid = CID[curve]
    bases = cv.g1.write_batch([cv.g1.gen] * 3, False)
    for bad in (cv.r, cv.r + 1, (1 << 760) - 1):  # 95 bytes hold values up to 2^760 - 1
        with pytest.raises(S.InvalidData) as ei:
            S.qap_dot_product(cid, 0, bases, False, [[(1, 0)], [(2, 1), (bad, 2)]], False)
        assert ei.value.index == 2
    with pytest.raises(S.InvalidLength):  # base index out of range
        S.qap_dot_product(cid, 0, bases, False, [[(1, 3)]], False)
