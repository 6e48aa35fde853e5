"""The ratio-check MSM (snark-setup_b200/csrc/msm.cuh: merge_pairs / power_pairs, setup-utils/src/helpers.rs:371-390)
against EXACT sums at the shapes production runs.

`sx == tau * s` cannot see a bug in the sort, the buckets or the reductions: s and sx go through the same stages, so such
a bug maps both by the same linear map and the relation still holds.  Here every input element has a known discrete
log, v_i = a_i * G, built on the device by apply_powers; the exact answer is then s = (sum rho_i a_i mod r) * G, which
costs O(n) integer work and one scalar multiplication at any n.  rho is either explicit or the device's own ChaCha20
scalars, restated by pyref_host.rho.  Results are compared byte for byte (uncompressed encodings).

Shapes: 2^21-pair tiles (c = 16, W = 8, 65 536 buckets per window) with a second tile of one pair; explicit scalars at
c = 11 (BLS12-377) and c = 14 (BW6-761); equal, cancelling and infinite inputs, which make the bucket sums small
multiples of one point; one bucket per window holding every point; and, one process per setting because the library
reads these variables once, every window width 2..16, tiny tiles, and the lane-split bucket accumulation."""
import functools
import operator
import os
import random
import subprocess
import sys

import pytest

import pyref as R
import pyref_host as H
import snark_setup_b200 as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T = 1 << 21                                  # default ratio tile (pairs per tile): api_ratio.inl ratio_tile_elems
SEED = bytes(range(7, 39))
CIDS = {"bls12_377": S.BLS12_377, "bw6_761": S.BW6_761, "mnt4_753": S.MNT4_753, "mnt6_753": S.MNT6_753}


# ---- ChaCha20 restatement (CPU) --------------------------------------------------------------------------------
def test_chacha20_blocks_match_the_scalar_block():
    rng = random.Random(1)
    key = bytes(rng.randrange(256) for _ in range(32))
    ctrs = [0, 1, 2, (1 << 32) - 2, (1 << 32) - 1, 1 << 32, (1 << 32) + 1] + [rng.randrange(1 << 40) for _ in range(4)]
    for c in ctrs:
        assert H.chacha20_blocks(key, c, 1)[0].tolist() == H.chacha20_block(key, c), c
    run = H.chacha20_blocks(key, (1 << 32) - 3, 6)  # a run crossing the 32-bit boundary of the counter
    assert [row.tolist() for row in run] == [H.chacha20_block(key, (1 << 32) - 3 + i) for i in range(6)]
    rho = H.rho(key, (1 << 32) - 1, 3)
    for i, v in enumerate(rho):
        w = H.chacha20_block(key, (1 << 32) - 1 + i)
        assert v == sum(w[k] << (32 * k) for k in range(4))


def test_chacha20_rfc8439_keystream_vectors():
    """RFC 8439 Appendix A.1, test vectors #1 and #2: key 0, nonce 0, block counters 0 and 1."""
    want = {0: "76b8e0ada0f13d90405d6ae55386bd28bdd219b8a08ded1aa836efcc8b770dc7"
               "da41597c5157488d7724e03fb8d84a376a43b8f41518a11cc387b669b2ee6586",
            1: "9f07e7be5551387a98ba977c732d080dcb0f29a048e3656912c6533e32ee7aed"
               "29b721769ce64e43d57133b074d839d531ed1f28510afb45ace10a1f4b794d6f"}
    for ctr, hx in want.items():
        assert b"".join(w.to_bytes(4, "little") for w in H.chacha20_block(bytes(32), ctr)).hex() == hx
        assert H.chacha20_blocks(bytes(32), ctr, 1)[0].astype("<u4").tobytes().hex() == hx
    assert H.rho(bytes(32), 0, 2) == [int.from_bytes(bytes.fromhex(want[c][:32]), "little") for c in (0, 1)]


# ---- inputs with known discrete logs -----------------------------------------------------------------------------
def _group(curve, gname):
    cv = R.curve_by_name(curve)
    return cv, getattr(cv, gname), CIDS[curve], S.G1 if gname == "g1" else S.G2


@functools.lru_cache(maxsize=4)
def _scalars(curve, kind, n, salt=0):
    """a_i of v_i = a_i * G: random, all 1 (equal points), 1 / r-1 alternating (P + (-P)), or random with runs of 0
    (runs of the point at infinity, one of them across the tile seam)."""
    r = R.curve_by_name(curve).r
    if kind == "ones":
        return [1] * n
    if kind == "alternating":
        return [1 if i % 2 == 0 else r - 1 for i in range(n)]
    rng = random.Random("%s/%s/%d/%d" % (curve, kind, n, salt))
    bits = r.bit_length() + 64
    a = [rng.getrandbits(bits) % r for _ in range(n)]
    if kind == "zero_runs":
        for i in range(n):
            if i % 1000 < 300 or abs(i - T) < 40:
                a[i] = 0
    return a


def _vector(curve, gname, a, compressed):
    """v_i = a_i * G through the device's apply_powers."""
    cv, g, cid, gid = _group(curve, gname)
    gens = g.encode(g.gen, True) * len(a)
    return S.apply_powers(cid, gid, gens, True, S.CHECK_NO, compressed, len(a), powers=a)


def _spot_check(curve, gname, a, buf, compressed, idx):
    """a wrong input vector must not hide a wrong MSM: v_i against pyref at the ends and the tile seam"""
    cv, g, _, _ = _group(curve, gname)
    sz = g.size(compressed)
    for i in sorted({i for i in idx if 0 <= i < len(a)}):
        assert buf[i * sz:(i + 1) * sz] == g.encode(g.mul(g.gen, a[i]), compressed), i


@functools.lru_cache(maxsize=2)
def _rho_seed(n):
    return H.rho(SEED, 0, n)


def _point(curve, gname, k):
    cv, g, _, _ = _group(curve, gname)
    return g.encode(g.mul(g.gen, k % cv.r), False)


def _want(curve, gname, rho, a1, a2):
    """(s, sx) = (sum rho_i a1_i, sum rho_i a2_i) * G over the pairs (len(rho) of them)"""
    return (_point(curve, gname, sum(map(operator.mul, rho, a1))), _point(curve, gname, sum(map(operator.mul, rho, a2))))


# ---- named cases: the parent computes the references, a child process under other settings the device results ----
# name -> (curve, group, op, n, scalars of v (or v1), scalars of v2 for merge_pairs)
CASES = {
    "power_bls_g2": ("bls12_377", "g2", "power", T + 2, "random", None),
    "merge_bls_g2": ("bls12_377", "g2", "merge", T + 1, "random", "random"),
    "ones_bls_g2": ("bls12_377", "g2", "power", T + 2, "ones", None),
    "alternating_bls_g2": ("bls12_377", "g2", "power", T + 2, "alternating", None),
    "zero_runs_bls_g2": ("bls12_377", "g2", "merge", T + 2, "zero_runs", "ones"),
    "ones_bls_g1": ("bls12_377", "g1", "power", T + 2, "ones", None),
    "alternating_bls_g1": ("bls12_377", "g1", "power", T + 2, "alternating", None),
    "zero_runs_bls_g1": ("bls12_377", "g1", "merge", T + 2, "zero_runs", "ones"),
}


def _case_inputs(name):
    curve, gname, op, n, k1, k2 = CASES[name]
    a1 = _scalars(curve, k1, n)
    a2 = _scalars(curve, k2, n, 1) if op == "merge" else None
    return curve, gname, op, n, a1, a2


def _case_device(name, spot_check=False):
    curve, gname, op, n, a1, a2 = _case_inputs(name)
    _, _, cid, gid = _group(curve, gname)
    v1 = _vector(curve, gname, a1, True)
    if spot_check:
        _spot_check(curve, gname, a1, v1, True, (0, 1, T - 1, T, n - 1))
    if op == "power":
        return S.power_pairs(cid, gid, v1, True, seed=SEED)
    return S.merge_pairs(cid, gid, v1, _vector(curve, gname, a2, True), True, seed=SEED)


def _case_want(name):
    curve, gname, op, n, a1, a2 = _case_inputs(name)
    if op == "power":
        return _want(curve, gname, _rho_seed(n - 1), a1[:-1], a1[1:])
    return _want(curve, gname, _rho_seed(n), a1, a2)


def _child(env, code):
    """run `code` in a fresh interpreter (the library reads its tuning variables once per process) -> stdout lines"""
    prelude = "import sys; sys.path[:0] = [%r, %r, %r]\n" % (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", prelude + code], env=dict(os.environ, **env), capture_output=True, text=True,
                       timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return r.stdout.split()


def _child_cases(env, names):
    code = ("import test_gpu_msm_reference as M\n"
            "for nm in %r:\n"
            "    s, sx = M._case_device(nm); print(nm, s.hex(), sx.hex())\n") % (list(names),)
    out = _child(env, code)
    return {out[i]: (bytes.fromhex(out[i + 1]), bytes.fromhex(out[i + 2])) for i in range(0, len(out), 3)}


# ---- generated rho at the production shape -----------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("curve,gname", [("bls12_377", "g1"), ("bls12_377", "g2"), ("bw6_761", "g1"), ("bw6_761", "g2")])
def test_generated_rho_production_shape(curve, gname):
    """power_pairs on 2^21 + 2 elements (one full tile, then one pair across the seam), check_and_ratio on the same
    vector with its re-emitted copy, merge_pairs on 2^21 + 1 pairs, and the swap of elements T-1 and T."""
    cv, g, cid, gid = _group(curve, gname)
    n = T + 2
    a = _scalars(curve, "random", n)
    vc = _vector(curve, gname, a, True)
    vu = _vector(curve, gname, a, False)
    seam = (0, 1, T - 2, T - 1, T, T + 1)
    _spot_check(curve, gname, a, vc, True, seam)
    _spot_check(curve, gname, a, vu, False, seam)
    rho = _rho_seed(n - 1)
    want = _want(curve, gname, rho, a[:-1], a[1:])
    assert S.power_pairs(cid, gid, vc, True, seed=SEED) == want
    out, s, sx = S.check_and_ratio(cid, gid, vc, True, seed=SEED, out_compressed=False)
    assert (s, sx) == want
    assert out == vu
    # merge_pairs(v[:T + 1], w): an independent second vector
    b = _scalars(curve, "random", T + 1, 1)
    w = _vector(curve, gname, b, False)
    _spot_check(curve, gname, b, w, False, (0, T - 1, T))
    assert S.merge_pairs(cid, gid, vu[:(T + 1) * g.usize], w, False, seed=SEED) == _want(curve, gname, rho, a[:T + 1], b)
    # swap the elements on both sides of the seam
    cs = g.csize
    sw = bytearray(vc)
    sw[(T - 1) * cs:T * cs], sw[T * cs:(T + 1) * cs] = vc[T * cs:(T + 1) * cs], vc[(T - 1) * cs:T * cs]
    a2 = list(a)
    a2[T - 1], a2[T] = a[T], a[T - 1]
    assert S.power_pairs(cid, gid, bytes(sw), True, seed=SEED) == _want(curve, gname, rho, a2[:-1], a2[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("curve", ["mnt4_753", "mnt6_753"])
@pytest.mark.parametrize("gname", ["g1", "g2"])
def test_generated_rho_mnt(curve, gname):
    """the 753-bit curves (G2 over Fq2 / Fq3): 2^14 + 1 pairs, tuned window 10, rounded to c = 8"""
    cv, g, cid, gid = _group(curve, gname)
    n = (1 << 14) + 2
    a = _scalars(curve, "random", n)
    vc = _vector(curve, gname, a, True)
    _spot_check(curve, gname, a, vc, True, (0, n // 2, n - 1))
    rho = _rho_seed(n - 1)
    assert S.power_pairs(cid, gid, vc, True, seed=SEED) == _want(curve, gname, rho, a[:-1], a[1:])


# ---- explicit rho at production widths ---------------------------------------------------------------------------
def _explicit_rho(r, c, n, rng):
    """random scalars with the edge cases spread over the vector: 0, 1, r-1, 2^(bits-1), every c-bit digit 2^c - 1
    (the top one as large as r allows) and only the top window non-zero"""
    bits = r.bit_length()
    W = (bits + c - 1) // c
    top = c * (W - 1)
    low = (1 << top) - 1                      # every digit below the top window = 2^c - 1
    all_max = low + ((r - 1 - low) >> top << top)
    only_top = (r - 1) >> top << top
    special = [0, 1, r - 1, 1 << (bits - 1), all_max, only_top, 1 << top, (1 << c) - 1]
    assert all(0 <= x < r for x in special)
    rho = [rng.randrange(r) for _ in range(n)]
    for k, x in enumerate(special):
        rho[k] = x
        rho[n // 2 + k] = x
        rho[n - 1 - k] = x
    return rho


@pytest.mark.gpu
@pytest.mark.parametrize("curve,gname,c", [("bls12_377", "g1", 11), ("bls12_377", "g2", 11), ("bw6_761", "g1", 14),
                                           ("bw6_761", "g2", 14)])
def test_explicit_rho_production_width(curve, gname, c):
    """explicit scalars lower c from the tuned width until it (almost) divides the scalar field: 2^17 pairs -> 13 -> 11
    for 253 bits, 2^18 pairs -> 14 for 377 bits"""
    cv, g, cid, gid = _group(curve, gname)
    n = (1 << (17 if c == 11 else 18)) + 2
    a = _scalars(curve, "random", n)
    vu = _vector(curve, gname, a, False)
    _spot_check(curve, gname, a, vu, False, (0, n - 1))
    rho = _explicit_rho(cv.r, c, n - 1, random.Random(c))
    assert S.power_pairs(cid, gid, vu, False, rho=rho) == _want(curve, gname, rho, a[:-1], a[1:])


@pytest.mark.gpu
@pytest.mark.parametrize("curve,gname", [("bls12_377", "g1"), ("bls12_377", "g2"), ("bw6_761", "g1")])
def test_one_bucket_holds_everything(curve, gname):
    """explicit rho all equal, every digit non-zero: every window is a single run of all 2^14 - 1 pairs (msm_order puts
    runs longer than 255 in one bin)"""
    cv, g, cid, gid = _group(curve, gname)
    n = 1 << 14
    a = _scalars(curve, "random", n)
    vc = _vector(curve, gname, a, True)
    for x in ((1 << (cv.r.bit_length() - 1)) - 1, cv.r - 1):
        rho = [x] * (n - 1)
        assert S.power_pairs(cid, gid, vc, True, rho=rho) == _want(curve, gname, rho, a[:-1], a[1:])


# ---- exceptional additions ---------------------------------------------------------------------------------------
EXCEPTIONAL = ["ones_bls_g1", "alternating_bls_g1", "zero_runs_bls_g1", "ones_bls_g2", "alternating_bls_g2",
               "zero_runs_bls_g2"]


@pytest.mark.gpu
@pytest.mark.parametrize("name", EXCEPTIONAL)
def test_exceptional_additions(name):
    """equal points (jac_madd doubles), P + (-P) and runs of the point at infinity read with CHECK_NO: the bucket sums
    are small multiples of one point, so the reductions' additions meet P == Q and P == -Q"""
    assert _case_device(name, spot_check=True) == _case_want(name)


# ---- other settings, one process each ----------------------------------------------------------------------------
@pytest.mark.gpu
def test_window_width_sweep():
    """SS_MSM_C_OFFSET=0 with SS_MSM_C_MAX = 2 .. 16 on 2^16 + 2 elements.  Generated rho is rho_i = the first 128 bits
    of ChaCha20 block i whatever the window, so (s, sx) are the same bytes for every width and equal the reference;
    explicit scalars (every width the lowering leaves: 253 bits -> 2 or 11, 377 bits -> 2, 3, 6, 7, 9, 13, 14) too."""
    n = (1 << 16) + 2
    code = ("import random, test_gpu_msm_reference as M, snark_setup_b200 as S\n"
            "for curve, gname in (('bls12_377', 'g1'), ('bw6_761', 'g1')):\n"
            "    cv, g, cid, gid = M._group(curve, gname)\n"
            "    v = M._vector(curve, gname, M._scalars(curve, 'random', %d), True)\n"
            "    s, sx = S.power_pairs(cid, gid, v, True, rho=M._explicit_rho(cv.r, 2, %d, random.Random(5)))\n"
            "    print(s.hex(), sx.hex())\n"
            "    s, sx = S.power_pairs(cid, gid, v, True, seed=M.SEED)\n"
            "    print(s.hex(), sx.hex())\n") % (n, n - 1)
    want = []
    for curve in ("bls12_377", "bw6_761"):
        cv = R.curve_by_name(curve)
        a = _scalars(curve, "random", n)
        rho = _explicit_rho(cv.r, 2, n - 1, random.Random(5))
        for rh in (rho, _rho_seed(n - 1)):
            want += [x.hex() for x in _want(curve, "g1", rh, a[:-1], a[1:])]
    got = {k: _child({"SS_MSM_C_OFFSET": "0", "SS_MSM_C_MAX": str(k)}, code) for k in range(2, 17)}
    bad = [k for k in got if got[k] != want]
    assert not bad, "window widths %s disagree with the exact reference" % bad


@pytest.mark.gpu
def test_many_small_tiles():
    """SS_RATIO_TILE_LOG2=10: 5 full tiles and a last tile of ONE pair, for power_pairs, merge_pairs and
    check_and_ratio, generated and explicit rho"""
    n = 5 * 1024 + 2
    code = ("import random, test_gpu_msm_reference as M, snark_setup_b200 as S\n"
            "for curve, gname in (('bls12_377', 'g1'), ('bls12_377', 'g2'), ('bw6_761', 'g1')):\n"
            "    cv, g, cid, gid = M._group(curve, gname)\n"
            "    n = %d\n"
            "    v = M._vector(curve, gname, M._scalars(curve, 'random', n), True)\n"
            "    w = M._vector(curve, gname, M._scalars(curve, 'random', n - 1, 1), True)\n"
            "    rho = M._explicit_rho(cv.r, 2, n - 1, random.Random(7))\n"
            "    out, s, sx = S.check_and_ratio(cid, gid, v, True, seed=M.SEED, out_compressed=True)\n"
            "    assert out == v\n"
            "    for r in (S.power_pairs(cid, gid, v, True, seed=M.SEED), (s, sx), S.power_pairs(cid, gid, v, True, rho=rho),\n"
            "              S.merge_pairs(cid, gid, v[:(n - 1) * g.csize], w, True, seed=M.SEED)):\n"
            "        print(r[0].hex(), r[1].hex())\n") % n
    want = []
    for curve, gname in (("bls12_377", "g1"), ("bls12_377", "g2"), ("bw6_761", "g1")):
        cv = R.curve_by_name(curve)
        a, b = _scalars(curve, "random", n), _scalars(curve, "random", n - 1, 1)
        gen = _rho_seed(n - 1)
        for rh, a1, a2 in ((gen, a[:-1], a[1:]), (gen, a[:-1], a[1:]),
                           (_explicit_rho(cv.r, 2, n - 1, random.Random(7)), a[:-1], a[1:]), (gen, a[:-1], b)):
            want += [x.hex() for x in _want(curve, gname, rh, a1, a2)]
    assert _child({"SS_RATIO_TILE_LOG2": "10"}, code) == want


@pytest.mark.gpu
def test_lane_split_bucket_accumulation():
    """SS_PAIR_KERNELS=6 switches the BLS12-377 G2 bucket accumulation to its lane-split twin (kept as an A/B path):
    the production shape and the exceptional inputs must give the exact sums there too"""
    names = ["power_bls_g2", "merge_bls_g2", "ones_bls_g2", "alternating_bls_g2", "zero_runs_bls_g2"]
    got = _child_cases({"SS_PAIR_KERNELS": "6"}, names)
    for nm in names:
        assert got[nm] == _case_want(nm), nm
