"""prepare_phase2 and the QAP evaluation on MNT4-753 / MNT6-753 through the C ABI: the group IFFT `to_coeffs`, the H query,
Groth16Params::new + ::write (setup-utils/src/groth16_utils.rs:44-168) and the sparse dot products of
phase2/src/polynomial.rs:11-94, for G1 and G2 (over Fq2 / Fq3) of both curves, against oracle/pyref.py.

Where the oracle's own transform is too slow (753-bit double-and-add in Python), points with known discrete logs carry
the check: P_i = a_i G built by the device's apply_powers (itself pinned to pyref in test_gpu_mnt.py and spot-checked
here), and the expected coefficients are scalar_ifft(a)_j G."""
import functools
import hashlib
import os
import random
import sys

import pytest

import pyref as R
import snark_setup_b200 as S

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import gen_constants as G  # noqa: E402

R.FR_GENERATOR.update(G.MNT_FFT_GENERATOR)  # GENERATOR = 17 of both MNT scalar fields (tools/gen_constants.py)

pytestmark = pytest.mark.gpu
CID = {"mnt4_753": S.MNT4_753, "mnt6_753": S.MNT6_753}
GROUPS = [(c, grp) for c in CID for grp in (0, 1)]


def _group(curve, grp):
    cv = R.curve_by_name(curve)
    return cv, (cv.g2 if grp else cv.g1)


def _exceptional_inputs(g, n, rng):
    """few distinct points: identities, repeats and negations, so the butterflies meet P + P and P - P"""
    base = [g.mul(g.gen, rng.randrange(1, g.r)) for _ in range(2)]
    pts = [rng.choice(base + [None]) for _ in range(n)]
    pts[0], pts[1], pts[2], pts[3] = base[0], base[0], g.neg(base[0]), None
    return pts


@pytest.mark.parametrize("curve,grp", GROUPS)
@pytest.mark.parametrize("log_n", [2, 3, 4])
def test_group_ifft_matches_pyref(curve, grp, log_n):
    cv, g = _group(curve, grp)
    n = 1 << log_n
    rng = random.Random(1000 * log_n + 10 * CID[curve] + grp)
    for pts in (_exceptional_inputs(g, n, rng), [g.mul(g.gen, rng.randrange(1, cv.r)) for _ in range(n)]):
        want = R.group_ifft_fast(g, pts)
        if log_n == 2:
            assert want == R.group_ifft(g, pts)
        for cin, cout in ((False, True), (True, False)):
            got = S.group_ifft(CID[curve], grp, g.write_batch(pts, cin), cin, cout)
            assert got == g.write_batch(want, cout), (cin, cout)
    for special in ([None] * n, [g.gen] * n):  # all identity; all equal (every stage-0 butterfly doubles)
        assert S.group_ifft(CID[curve], grp, g.write_batch(special, False), False, True) == \
            g.write_batch(R.group_ifft_fast(g, special), True)


def _known_log_ifft(curve, grp, a, spot):
    """device group_ifft of a_i G against scalar_ifft(a)_j G, both vectors made by apply_powers"""
    cv, g = _group(curve, grp)
    cid, n = CID[curve], len(a)
    gens = g.encode(g.gen, True) * n
    pts = S.apply_powers(cid, grp, gens, True, S.CHECK_NO, False, n, powers=a)
    c = R.scalar_ifft(cv.r, a)
    want = S.apply_powers(cid, grp, gens, True, S.CHECK_NO, True, n, powers=c)
    sz, csz = g.size(False), g.size(True)
    for i in spot:  # the two reference vectors against the oracle's scalar multiplication
        assert pts[i * sz:(i + 1) * sz] == g.encode(g.mul(g.gen, a[i]), False), i
        assert want[i * csz:(i + 1) * csz] == g.encode(g.mul(g.gen, c[i]), True), i
    assert S.group_ifft(cid, grp, pts, False, True) == want


@pytest.mark.parametrize("curve,grp", GROUPS)
@pytest.mark.parametrize("log_n", [5, 6, 7, 8])
def test_group_ifft_known_discrete_logs(curve, grp, log_n):
    cv, _ = _group(curve, grp)
    n = 1 << log_n
    rng = random.Random(log_n * 7 + CID[curve] * 3 + grp)
    a = [rng.randrange(cv.r) for _ in range(n)]
    for i in range(0, n, 5):
        a[i] = 0  # identities
    for i in range(1, n, 7):
        a[i] = a[1]  # repeated points
    a[2] = cv.r - a[1]  # a negation
    _known_log_ifft(curve, grp, a, (1, 2, n - 1))


@pytest.mark.parametrize("curve", list(CID))
def test_group_ifft_large_g1(curve):
    cv, _ = _group(curve, 0)
    n = 1 << 12
    rng = random.Random(4096 + CID[curve])
    a = [rng.randrange(cv.r) for _ in range(n)]
    a[17] = 0
    _known_log_ifft(curve, 0, a, (0, 17, n // 2 + 3))


@functools.lru_cache(maxsize=2)
def _accumulator(curve, power):
    """a full Groth16 accumulator from pyref's Phase1::computation on the derived-generator blank (test input only:
    arkworks' MNT G2 generator is not known here)"""
    cv = R.curve_by_name(curve)
    rp = R.Phase1Parameters(cv, power, 256)
    sp = S.Phase1Parameters(CID[curve], power, 256)
    keys = [int.from_bytes(hashlib.blake2b(curve.encode() + bytes([i]), digest_size=64).digest(), "little") % (cv.r - 2) + 2
            for i in range(3)]
    acc = bytes(R.phase1_computation(rp, bytes(R.phase1_initialization(rp, False)), False, False, R.NO, *keys))
    return rp, sp, acc


@functools.lru_cache(maxsize=None)
def _pyref_ifft(g, pts):
    return R.group_ifft_fast(g, list(pts))


def _pyref_params(rp, acc, phase2_size, cout):
    return R.groth16_params_new(rp, acc, False, phase2_size, cout, ifft=lambda g, pts: _pyref_ifft(g, tuple(pts)))


POWER = 6


@pytest.mark.parametrize("curve", list(CID))
def test_h_query_on_accumulator(curve):
    cv = R.curve_by_name(curve)
    rp, sp, acc = _accumulator(curve, POWER)
    o, c, s = rp.split_offsets(False)[0]
    tau_g1 = acc[o:o + c * s]
    pts = cv.g1.read_batch(tau_g1, False)
    for degree in (1, 2, 1 << POWER):
        for cout in (False, True):
            got = S.h_query_groth16(CID[curve], tau_g1, False, degree, cout)
            assert got == cv.g1.write_batch(R.h_query_groth16(cv.g1, pts, degree), cout), (degree, cout)


@pytest.mark.parametrize("curve", list(CID))
def test_groth16_params_new_matches_pyref(curve):
    rp, sp, acc = _accumulator(curve, POWER)
    for phase2_size in (1 << POWER, 5):
        for cout in (False, True):
            got = S.groth16_params_new(sp, acc, False, phase2_size, cout)
            assert got == _pyref_params(rp, acc, phase2_size, cout), (phase2_size, cout)
    # compressed accumulator in, read with full validation
    acc_c = bytearray(sp.get_length(True))
    acc_c[:64] = acc[:64]
    for (o, c, s), (oc, _, sc), grp in zip(rp.split_offsets(False), rp.split_offsets(True), (0, 1, 0, 0, 1)):
        acc_c[oc:oc + c * sc] = S.transcode(CID[curve], grp, acc[o:o + c * s], False, S.CHECK_NO, True)
    got = S.groth16_params_new(sp, bytes(acc_c), True, 1 << POWER, True, check=S.CHECK_FULL)
    assert got == _pyref_params(rp, acc, 1 << POWER, True)
    with pytest.raises(S.InvalidLength):  # domain larger than the powers of tau
        S.groth16_params_new(sp, acc, False, (1 << POWER) + 1, False)


def _rows(rng, r, num_vars, n_bases):
    rows = []
    for _ in range(num_vars):
        rows.append([(rng.choice([1, r - 1, 1, r - 1, 2, rng.randrange(r), 0]), rng.randrange(n_bases))
                     for _ in range(rng.randrange(0, 4))])
    return rows


@pytest.mark.parametrize("curve,grp", GROUPS)
def test_dot_product_vec_matches_pyref(curve, grp):
    cv, g = _group(curve, grp)
    rng = random.Random(70 + 2 * CID[curve] + grp)
    n = 10
    bases = [g.mul(g.gen, rng.randrange(1, cv.r)) for _ in range(n)]
    bases[5] = None
    rows = _rows(rng, cv.r, 16, n)
    rows[0] = [(rng.choice([1, cv.r - 1, rng.randrange(cv.r)]), i) for i in range(n)] * 3  # one dense row
    rows[3] = []                                        # empty rows -> infinity
    rows[9] = []
    rows[4] = [(1, 2), (cv.r - 1, 2)]                   # cancels
    rows[6] = [(1, 7), (1, 7)]                          # doubling inside the sum
    rows[7] = [(5, 1), (cv.r - 5, 1)]                   # general entries cancelling
    rows[8] = [(3, 4), (3, 4), (cv.r - 1, 8)]           # equal general entries: P + P of Jacobian sums
    want = R.dot_product_vec(g, rows, bases)
    for cin, cout in ((False, True), (True, False)):
        got = S.qap_dot_product(CID[curve], grp, g.write_batch(bases, cin), cin, rows, cout)
        assert got == g.write_batch(want, cout)


@pytest.mark.parametrize("curve", list(CID))
def test_qap_eval_small_circuit(curve):
    """polynomial.rs:11-47 on a toy QAP: a/b/c matrices over 4 constraints and 5 variables (2 public)."""
    cv, cid = R.curve_by_name(curve), CID[curve]
    g1, g2 = cv.g1, cv.g2
    rng = random.Random(5 + cid)
    m, num_vars, num_inputs = 4, 5, 2
    co1 = [g1.mul(g1.gen, rng.randrange(1, cv.r)) for _ in range(m)]
    co2 = [g2.mul(g2.gen, rng.randrange(1, cv.r)) for _ in range(m)]
    al = [g1.mul(g1.gen, rng.randrange(1, cv.r)) for _ in range(m)]
    be = [g1.mul(g1.gen, rng.randrange(1, cv.r)) for _ in range(m)]

    def matrix():
        return [[(rng.choice([1, cv.r - 1, rng.randrange(cv.r)]), rng.randrange(num_vars)) for _ in range(rng.randrange(1, 4))]
                for _ in range(m)]
    at, bt, ct = (R.process_matrix(matrix(), num_vars) for _ in range(3))
    a_g1, b_g1, b_g2, gamma_abc, l = R.qap_eval(cv, co1, co2, al, be, at, bt, ct, num_inputs)
    b1 = g1.write_batch(co1, False)
    assert S.qap_dot_product(cid, 0, b1, False, at, False) == g1.write_batch(a_g1, False)
    assert S.qap_dot_product(cid, 0, b1, False, bt, True) == g1.write_batch(b_g1, True)
    assert S.qap_dot_product(cid, 1, g2.write_batch(co2, True), True, bt, False) == g2.write_batch(b_g2, False)
    ext_rows = [[(c, i) for c, i in a] + [(c, i + m) for c, i in b] + [(c, i + 2 * m) for c, i in cc]
                for a, b, cc in zip(at, bt, ct)]
    ext = S.qap_dot_product(cid, 0, g1.write_batch(be + al + co1, False), False, ext_rows, False)
    assert ext == g1.write_batch(gamma_abc + l, False)
