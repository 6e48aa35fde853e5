"""Phase-2 contribute and verify as engine calls (MPCParameters::contribute / verify, phase2/src/parameters.rs:286-411)
on the H and L queries, against pyref, against the primitive composition they replace (transcode -> batch_mul ->
transcode; merge_pairs), and against exact sums.

Query elements have known discrete logs, v_i = a_i * G, built on the device by apply_powers, so the expected contribute
output (a_i / delta) * G and the expected verification pairs (sum rho_i a_i) * G cost O(n) integer work at any n; pyref
checks a sample of elements directly.  Sizes 1, 2^10 + 3 and 2^21 + 1 (which crosses the 1 212 416-element contribute
tile and the 2^21-pair ratio tile)."""
import random

import pytest

import pyref as R
import pyref_host as H
import snark_setup_b200 as S
from snark_setup_b200 import ffi

pytestmark = pytest.mark.gpu

SEED = bytes(range(3, 35))
CURVES = {"bls12_377": (R.BLS12_377, S.BLS12_377), "bw6_761": (R.BW6_761, S.BW6_761)}
BIG = (1 << 21) + 1


@pytest.fixture(params=[True, False], ids=["concurrent", "sequential"])
def concurrent(request):
    ffi.set_concurrent_vectors(request.param)
    yield request.param
    ffi.set_concurrent_vectors(True)


def _points(cid, g, a, compressed):
    """a_i * G, serialized with `compressed`, through the device's apply_powers"""
    return S.apply_powers(cid, S.G1, g.encode(g.gen, True) * len(a), True, S.CHECK_NO, compressed, len(a), powers=a)


def _dlogs(cv, n, salt, zeros=()):
    rng = random.Random("%s/%d/%s" % (cv.name, n, salt))
    a = [rng.randrange(1, cv.r) for _ in range(n)]
    for i in zeros:
        if i < n:
            a[i] = 0  # the point at infinity
    return a


def _elem(buf, i, sz):
    return bytes(buf[i * sz:(i + 1) * sz])


def _batch_mul_composition(cid, q, compressed, coeff):
    """what a caller composes today: transcode -> batch_mul -> transcode"""
    u = bytearray(S.transcode(cid, S.G1, q, compressed, S.CHECK_NO, False)) if compressed else bytearray(q)
    S.batch_mul(cid, S.G1, u, coeff)
    return S.transcode(cid, S.G1, bytes(u), False, S.CHECK_NO, True) if compressed else bytes(u)


# ---- contribute --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("compressed", [True, False], ids=["compressed", "uncompressed"])
@pytest.mark.parametrize("curve", list(CURVES))
def test_contribute_matches_pyref_and_batch_mul(curve, compressed):
    cv, cid = CURVES[curve]
    g1, g2 = cv.g1, cv.g2
    sz = S.element_size(cid, S.G1, compressed)
    rng = random.Random(curve)
    for n in (1, (1 << 10) + 3):
        a_h, a_l = _dlogs(cv, n, "h", zeros=(0, 5)), _dlogs(cv, n + 1, "l", zeros=(n,))
        h0, l0 = _points(cid, g1, a_h, compressed), _points(cid, g1, a_l, compressed)
        for delta in (1, 2, cv.r - 1, rng.randrange(2, cv.r)):
            inv = pow(delta, -1, cv.r)
            d1 = g1.mul(g1.gen, rng.randrange(1, cv.r))
            d2 = g2.mul(g2.gen, rng.randrange(1, cv.r))
            h, l = bytearray(h0), bytearray(l0)
            e1, e2 = bytearray(g1.encode(d1, compressed)), bytearray(g2.encode(d2, compressed))
            S.phase2_contribute(cid, delta, h, l, compressed, S.CHECK_NO, e1, e2)
            assert bytes(h) == _points(cid, g1, [x * inv % cv.r for x in a_h], compressed), (n, delta)
            assert bytes(l) == _points(cid, g1, [x * inv % cv.r for x in a_l], compressed), (n, delta)
            assert bytes(h) == _batch_mul_composition(cid, h0, compressed, inv)
            assert bytes(l) == _batch_mul_composition(cid, l0, compressed, inv)
            for i in sorted({0, n - 1, n // 2, 5 % n}):
                assert _elem(h, i, sz) == g1.encode(g1.mul(g1.mul(g1.gen, a_h[i]), inv), compressed), (n, delta, i)
            assert _elem(l, n, sz) == g1.encode(None, compressed)  # the identity stays the identity
            assert bytes(e1) == g1.encode(g1.mul(d1, delta), compressed)
            assert bytes(e2) == g2.encode(g2.mul(d2, delta), compressed)


@pytest.mark.parametrize("compressed", [True, False], ids=["compressed", "uncompressed"])
@pytest.mark.parametrize("curve", list(CURVES))
def test_contribute_across_tiles(curve, compressed):
    """2^21 + 1 and 2^21 elements: exact (delta^-1 tau^i) * G from apply_powers, and the primitive composition"""
    cv, cid = CURVES[curve]
    g1 = cv.g1
    rng = random.Random("big/" + curve)
    tau, delta = rng.randrange(2, cv.r), rng.randrange(2, cv.r)
    inv = pow(delta, -1, cv.r)
    gens = g1.encode(g1.gen, True)
    q = {n: S.apply_powers(cid, S.G1, gens * n, True, S.CHECK_NO, compressed, n, tau=tau, first_power=f)
         for n, f in ((BIG, 0), (BIG - 1, 3))}
    h, l = bytearray(q[BIG]), bytearray(q[BIG - 1])
    S.phase2_contribute(cid, delta, h, l, compressed, S.CHECK_NO)
    for buf, n, f in ((h, BIG, 0), (l, BIG - 1, 3)):
        want = S.apply_powers(cid, S.G1, gens * n, True, S.CHECK_NO, compressed, n, tau=tau, first_power=f, coeff=inv)
        assert bytes(buf) == want, n
    assert bytes(h) == _batch_mul_composition(cid, q[BIG], compressed, inv)


@pytest.mark.parametrize("curve", list(CURVES))
def test_contribute_shards_equal_the_whole_call(curve, concurrent):
    cv, cid = CURVES[curve]
    g1, g2 = cv.g1, cv.g2
    rng = random.Random("shard/" + curve)
    delta = rng.randrange(2, cv.r)
    for n_h, n_l in ((5, 6), ((1 << 10) + 3, 700)):
        h0 = _points(cid, g1, _dlogs(cv, n_h, "sh"), True)
        l0 = _points(cid, g1, _dlogs(cv, n_l, "sl"), True)
        d10, d20 = g1.encode(g1.mul(g1.gen, 11), True), g2.encode(g2.mul(g2.gen, 13), True)
        h, l, d1, d2 = bytearray(h0), bytearray(l0), bytearray(d10), bytearray(d20)
        S.phase2_contribute(cid, delta, h, l, True, S.CHECK_NO, d1, d2)
        for count in (1, 3, 8):
            hs, ls, e1, e2 = bytearray(h0), bytearray(l0), bytearray(d10), bytearray(d20)
            for k in range(count):
                S.phase2_contribute(cid, delta, hs, ls, True, S.CHECK_NO, e1, e2, shard=(k, count))
            assert (hs, ls, e1, e2) == (h, l, d1, d2), (n_h, count)


@pytest.mark.parametrize("curve", list(CURVES))
def test_contribute_errors_name_the_query(curve, concurrent):
    """a bad element is reported with its query-relative index and the query's name; H wins when both are bad"""
    cv, cid = CURVES[curve]
    g1 = cv.g1
    sz = S.element_size(cid, S.G1, True)
    h0, l0 = _points(cid, g1, _dlogs(cv, 40, "eh"), True), _points(cid, g1, _dlogs(cv, 30, "el"), True)
    inf = g1.encode(None, True)

    def bad(q, i):
        b = bytearray(q)
        b[i * sz:(i + 1) * sz] = inf
        return b
    for h, l, idx, name in ((bad(h0, 17), bytearray(l0), 17, "h_query"), (bytearray(h0), bad(l0, 29), 29, "l_query"),
                            (bad(h0, 33), bad(l0, 2), 33, "h_query")):
        with pytest.raises(S.PointAtInfinity) as ei:
            S.phase2_contribute(cid, 5, h, l, True, S.CHECK_ONLY_NON_ZERO)
        assert ei.value.index == idx and name in str(ei.value), (idx, name, ei.value.index, str(ei.value))
    # the shard that owns the element reports it with the query-relative index
    with pytest.raises(S.PointAtInfinity) as ei:
        S.phase2_contribute(cid, 5, bytearray(h0), bad(l0, 29), True, S.CHECK_ONLY_NON_ZERO, shard=(2, 3))
    assert ei.value.index == 29 and "l_query" in str(ei.value)


# ---- verification pairs ------------------------------------------------------------------------------------------
def _exact_pairs(cv, seed, a_before, a_after, first=0):
    g = cv.g1
    rho = H.rho(seed, first, len(a_before))
    s = sum(x * y for x, y in zip(rho, a_before)) % cv.r
    sx = sum(x * y for x, y in zip(rho, a_after)) % cv.r
    return g.encode(g.mul(g.gen, s), False), g.encode(g.mul(g.gen, sx), False)


@pytest.mark.parametrize("curve", list(CURVES))
def test_verification_pairs_are_exact_and_shard(curve, concurrent):
    cv, cid = CURVES[curve]
    g1 = cv.g1
    rng = random.Random("pairs/" + curve)
    delta = rng.randrange(2, cv.r)
    inv = pow(delta, -1, cv.r)
    n_h, n_l = (BIG, (1 << 10) + 3) if concurrent else (1000, 7)
    for compressed in (True, False):
        a_h, a_l = _dlogs(cv, n_h, "ph"), _dlogs(cv, n_l, "pl", zeros=(3,))
        hb, lb = _points(cid, g1, a_h, compressed), _points(cid, g1, a_l, compressed)
        ha, la = bytearray(hb), bytearray(lb)
        S.phase2_contribute(cid, delta, ha, la, compressed)
        # CHECK_NO: the L query holds the point at infinity, which merge_pairs sums like any other point
        pairs = lambda shard=None: S.phase2_verification_pairs(cid, hb, ha, lb, la, compressed, S.CHECK_NO, S.CHECK_NO,  # noqa: E731
                                                               seed=SEED, shard=shard, raw=True)
        whole = pairs()
        u = S.element_size(cid, S.G1, False)
        got = [whole[k * u:(k + 1) * u] for k in range(4)]
        want = _exact_pairs(cv, SEED, a_h, [x * inv % cv.r for x in a_h]) + \
            _exact_pairs(cv, SEED, a_l, [x * inv % cv.r for x in a_l])
        assert got == list(want), (compressed, n_h)
        # merge_pairs(before, after) composed from the primitive gives the same pairs
        if n_h < BIG:
            assert S.merge_pairs(cid, S.G1, hb, bytes(ha), compressed, seed=SEED) == (got[0], got[1])
        for count in (3, 8):
            parts = [pairs((k, count)) for k in range(count)]
            assert S.phase2_reduce_partial_pairs(cid, parts, raw=True) == whole, count


# ---- verdicts ----------------------------------------------------------------------------------------------------
def _round(curve, compressed, n_h=300, n_l=200):
    """one honest contribution: (before h, l), (after h, l), delta_g1_after, delta_g2_before, delta_g2_after"""
    cv, cid = CURVES[curve]
    g1, g2 = cv.g1, cv.g2
    rng = random.Random("round/%s/%s" % (curve, compressed))
    d_prev, delta = rng.randrange(2, cv.r), rng.randrange(2, cv.r)
    hb = _points(cid, g1, _dlogs(cv, n_h, "vh"), compressed)
    lb = _points(cid, g1, _dlogs(cv, n_l, "vl"), compressed)
    ha, la = bytearray(hb), bytearray(lb)
    d1 = bytearray(g1.encode(g1.mul(g1.gen, d_prev), compressed))
    d2b = g2.encode(g2.mul(g2.gen, d_prev), compressed)
    d2 = bytearray(d2b)
    S.phase2_contribute(cid, delta, ha, la, compressed, S.CHECK_NO, d1, d2)
    return cv, cid, hb, bytes(ha), lb, bytes(la), bytes(d1), d2b, bytes(d2)


def _verify(r, hb=None, ha=None, lb=None, la=None, d1=None, d2b=None, d2a=None, compressed=True, **kw):
    cv, cid, hb0, ha0, lb0, la0, d10, d2b0, d2a0 = r
    S.phase2_verification(cid, hb or hb0, ha or ha0, lb or lb0, la or la0, compressed, d1 or d10, d2b or d2b0,
                          d2a or d2a0, seed=SEED, **kw)


def _put(buf, i, sz, enc):
    b = bytearray(buf)
    b[i * sz:(i + 1) * sz] = enc
    return bytes(b)


def _off_subgroup_point(g, rng):
    F = g.F
    while True:
        x = rng.randrange(F.p)
        y = F.sqrt(F.add(F.mul(F.sqr(x), x), g.b))
        if y is not None and not g.in_subgroup((x, y)):
            return (x, y)


@pytest.mark.parametrize("compressed", [True, False], ids=["compressed", "uncompressed"])
@pytest.mark.parametrize("curve", list(CURVES))
def test_verification_verdicts(curve, compressed):
    r = _round(curve, compressed)
    cv, cid, hb, ha, lb, la, d1, d2b, d2a = r
    g1, g2 = cv.g1, cv.g2
    sz = S.element_size(cid, S.G1, compressed)
    v = lambda **kw: _verify(r, compressed=compressed, **kw)  # noqa: E731
    v()
    v(check_before=S.CHECK_FULL, check_after=S.CHECK_FULL)

    def ratio_fails(index, **kw):
        with pytest.raises(S.InvalidRatio) as ei:
            v(**kw)
        assert ei.value.index == index, (index, ei.value.index, str(ei.value))
        assert ["delta", "h_query", "l_query"][index] in str(ei.value)

    swapped = _put(_put(ha, 10, sz, _elem(ha, 11, sz)), 11, sz, _elem(ha, 10, sz))
    ratio_fails(1, ha=swapped)
    ratio_fails(2, lb=_put(lb, 50, sz, g1.encode(g1.mul(g1.gen, 12345), compressed)))
    ratio_fails(0, d2a=g2.encode(g2.mul(g2.gen, 777), compressed))
    ratio_fails(1, ha=swapped, lb=_put(lb, 50, sz, g1.encode(g1.gen, compressed)))  # H before L

    # an off-subgroup point in `after`: the subgroup pass reports it with its L index (Full: the decoder's InvalidData)
    off = g1.encode(_off_subgroup_point(g1, random.Random(curve)), compressed)
    with pytest.raises(S.IncorrectSubgroup) as ei:
        v(la=_put(la, 123, sz, off), check_after=S.CHECK_ONLY_NON_ZERO)
    assert ei.value.index == 123 and "l_query" in str(ei.value)
    with pytest.raises(S.InvalidData) as ei:
        v(la=_put(la, 123, sz, off), check_after=S.CHECK_FULL)
    assert ei.value.index == 123
    with pytest.raises(S.InvalidData):  # as ss_transcode reports it
        S.transcode(cid, S.G1, _put(la, 123, sz, off), compressed, S.CHECK_FULL, False)
    # the same point in `before`, read with No, gets no subgroup test: only the ratio fails
    ratio_fails(2, lb=_put(lb, 123, sz, off), check_before=S.CHECK_NO, check_after=S.CHECK_ONLY_NON_ZERO)
    # ... and a bad element in both queries is reported in H
    with pytest.raises(S.IncorrectSubgroup) as ei:
        v(ha=_put(ha, 7, sz, off), la=_put(la, 3, sz, off), check_after=S.CHECK_ONLY_NON_ZERO)
    assert ei.value.index == 7 and "h_query" in str(ei.value)

    inf = g1.encode(None, compressed)
    for check in (S.CHECK_ONLY_NON_ZERO, S.CHECK_FULL):
        with pytest.raises(S.PointAtInfinity) as ei:
            v(ha=_put(ha, 299, sz, inf), check_after=check)
        assert ei.value.index == 299 and "h_query" in str(ei.value)


@pytest.mark.parametrize("curve", list(CURVES))
def test_check_ratio_pairs_from_reduced_shards(curve):
    r = _round(curve, True)
    cv, cid, hb, ha, lb, la, d1, d2b, d2a = r
    parts = [S.phase2_verification_pairs(cid, hb, ha, lb, la, True, seed=SEED, shard=(k, 3), raw=True) for k in range(3)]
    pairs = S.phase2_reduce_partial_pairs(cid, parts, raw=True)
    unc = lambda g, b: S.transcode(cid, g, b, True, S.CHECK_NO, False)  # noqa: E731
    S.phase2_check_ratio_pairs(cid, pairs, unc(S.G1, d1), unc(S.G2, d2b), unc(S.G2, d2a))
    # a wrong delta_g2_before leaves the delta check (index 0) valid and fails H, the first check that reads it
    with pytest.raises(S.InvalidRatio) as ei:
        S.phase2_check_ratio_pairs(cid, pairs, unc(S.G1, d1), unc(S.G2, d2a), unc(S.G2, d2a))
    assert ei.value.index == 1


def test_empty_query_is_batch_too_small():
    r = _round("bls12_377", True, 4, 4)
    cv, cid, hb, ha, lb, la, d1, d2b, d2a = r
    with pytest.raises(ffi.BatchTooSmall):
        S.phase2_verification(cid, hb, ha, b"", b"", True, d1, d2b, d2a, seed=SEED)


# ---- MNT4-753 / MNT6-753 -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["mnt4_753", "mnt6_753"])
def test_mnt_contribute_and_pairs_match_pyref(name):
    cv = R.curve_by_name(name)
    cid = {"mnt4_753": S.MNT4_753, "mnt6_753": S.MNT6_753}[name]
    g1, g2 = cv.g1, cv.g2
    n = 1 << 8
    rng = random.Random(name)
    delta = rng.randrange(2, cv.r)
    inv = pow(delta, -1, cv.r)
    a_h, a_l = _dlogs(cv, n, "mh"), _dlogs(cv, n, "ml")
    hb, lb = _points(cid, g1, a_h, True), _points(cid, g1, a_l, True)
    ha, la = bytearray(hb), bytearray(lb)
    p2 = g2.mul(g2.gen, 5)
    d2 = bytearray(g2.encode(p2, True))
    S.phase2_contribute(cid, delta, ha, la, True, S.CHECK_NO, None, d2)
    assert bytes(ha) == _points(cid, g1, [x * inv % cv.r for x in a_h], True)
    assert bytes(la) == _points(cid, g1, [x * inv % cv.r for x in a_l], True)
    sz = S.element_size(cid, S.G1, True)
    for i in (0, 77, n - 1):
        assert _elem(ha, i, sz) == g1.encode(g1.mul(g1.gen, a_h[i] * inv % cv.r), True)
    assert bytes(d2) == g2.encode(g2.mul(p2, delta), True)
    got = S.phase2_verification_pairs(cid, hb, bytes(ha), lb, bytes(la), True, seed=SEED, raw=True)
    u = S.element_size(cid, S.G1, False)
    want = _exact_pairs(cv, SEED, a_h, [x * inv % cv.r for x in a_h]) + \
        _exact_pairs(cv, SEED, a_l, [x * inv % cv.r for x in a_l])
    assert [got[k * u:(k + 1) * u] for k in range(4)] == list(want)
    with pytest.raises(S.InvalidArgument):
        S.phase2_check_ratio_pairs(cid, got, bytes(u), bytes(2 * u), bytes(2 * u))
