"""Phase-2 contribute / verify entry points without a device: blob sizes, and the argument checks that run before any
device is touched (null pointers, bad enums, delta = 0 or >= r, shard arguments, MNT pairing checks)."""
import ctypes as C

import pytest

import pyref as R
import snark_setup_b200 as S
from snark_setup_b200 import ffi

CURVES = [(S.BLS12_377, R.BLS12_377), (S.BW6_761, R.BW6_761), (S.MNT4_753, None), (S.MNT6_753, None)]
SEED = bytes(range(32))


def _g1(cid, compressed=False):
    return bytes(S.element_size(cid, S.G1, compressed))


def _contribute(cid, delta, h=None, l=None, compressed=False, check=S.CHECK_NO, shard=(0, 1)):
    """the raw call, so that NULL and out-of-range arguments can be passed"""
    f = S.lib().ss_phase2_contribute_shard
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                  C.c_void_p, C.c_uint32, C.c_uint32]
    sz = max(1, S.element_size(cid, S.G1, compressed))
    return f(cid, delta, h, len(h or b"") // sz, l, len(l or b"") // sz, int(compressed), check, None, None, *shard)


def _pairs(cid, n=2, seed=SEED, check_before=S.CHECK_NO, check_after=S.CHECK_NO, subgroup=0, shard=(0, 1), null_q=False,
           out=True):
    f = S.lib().ss_phase2_verification_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_size_t, C.c_char_p, C.c_char_p, C.c_size_t, C.c_int, C.c_int,
                  C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]
    q = None if null_q else _g1(cid) * n
    buf = C.create_string_buffer(max(1, ffi.phase2_pairs_size(cid))) if out else None
    return f(cid, q, q, n, q, q, n, 0, check_before, check_after, subgroup, seed, buf, *shard)


def _code(rc):
    return ffi._ERRORS.get(rc) if rc else None


@pytest.mark.parametrize("cid,cv", CURVES, ids=["bls12_377", "bw6_761", "mnt4_753", "mnt6_753"])
def test_pairs_size_is_four_uncompressed_g1(cid, cv):
    assert ffi.phase2_pairs_size(cid) == 4 * S.element_size(cid, S.G1, False)
    if cv is not None:
        assert ffi.phase2_pairs_size(cid) == 4 * len(cv.g1.encode(cv.g1.gen, False))
    assert ffi.phase2_pairs_size(7) == 0


@pytest.mark.parametrize("cid,cv", CURVES[:2], ids=["bls12_377", "bw6_761"])
def test_contribute_rejects_bad_arguments_before_the_device(cid, cv):
    fb = S.scalar_size(cid)
    good = (5).to_bytes(fb, "little")
    q = _g1(cid) * 2
    bad = {
        "delta = 0": _contribute(cid, bytes(fb), q, q),
        "delta = r": _contribute(cid, cv.r.to_bytes(fb, "little"), q, q),
        "delta = 2^bits - 1": _contribute(cid, b"\xff" * fb, q, q),
        "null delta": _contribute(cid, None, q, q),
        "null query": S.lib().ss_phase2_contribute(cid, good, None, 2, None, 0, 0, 3, None, None),
        "bad check": _contribute(cid, good, q, q, check=4),
        "negative check": _contribute(cid, good, q, q, check=-1),
        "unknown curve": _contribute(9, good, q, q),
        "shard count 0": _contribute(cid, good, q, q, shard=(0, 0)),
        "shard index >= count": _contribute(cid, good, q, q, shard=(3, 3)),
    }
    assert {k: _code(v) for k, v in bad.items()} == {k: S.InvalidArgument for k in bad}
    # valid arguments get as far as the device: without one that is a DeviceError, never a CPU result
    assert _code(_contribute(cid, (cv.r - 1).to_bytes(fb, "little"), q, q)) in (S.DeviceError, None)


@pytest.mark.parametrize("cid", [S.BLS12_377, S.BW6_761, S.MNT4_753, S.MNT6_753])
def test_verification_pairs_rejects_bad_arguments_before_the_device(cid):
    bad = {
        "null seed": _pairs(cid, seed=None),
        "null pairs": _pairs(cid, out=False),
        "null queries": _pairs(cid, null_q=True),
        "bad check_before": _pairs(cid, check_before=4),
        "bad check_after": _pairs(cid, check_after=-1),
        "bad subgroup mode": _pairs(cid, subgroup=4),
        "shard index >= count": _pairs(cid, shard=(2, 2)),
        "unknown curve": _pairs(5),
    }
    assert {k: _code(v) for k, v in bad.items()} == {k: S.InvalidArgument for k in bad}
    assert _code(_pairs(cid, n=0)) is ffi.BatchTooSmall  # an empty whole query, as ss_merge_pairs
    rc = S.lib().ss_phase2_reduce_partial_pairs(cid, None, 1, None)
    assert _code(rc) is S.InvalidArgument


@pytest.mark.parametrize("cid", [S.MNT4_753, S.MNT6_753])
def test_mnt_has_no_device_verdict(cid):
    u1, u2 = S.element_size(cid, S.G1, False), S.element_size(cid, S.G2, False)
    with pytest.raises(S.InvalidArgument, match="no device pairing"):
        ffi.phase2_check_ratio_pairs(cid, bytes(4 * u1), bytes(u1), bytes(u2), bytes(u2))
    # refused before any query is read: the queries passed here are not even valid encodings
    q = b"\xff" * (2 * S.element_size(cid, S.G1, True))
    c1, c2 = S.element_size(cid, S.G1, True), S.element_size(cid, S.G2, True)
    with pytest.raises(S.InvalidArgument, match="no device pairing"):
        ffi.phase2_verification(cid, q, q, q, q, True, bytes(c1), bytes(c2), bytes(c2), seed=SEED)


def test_check_ratio_pairs_rejects_null_arguments():
    u1 = S.element_size(S.BLS12_377, S.G1, False)
    f = S.lib().ss_phase2_check_ratio_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
    assert _code(f(S.BLS12_377, None, bytes(u1), bytes(2 * u1), bytes(2 * u1))) is S.InvalidArgument
    assert _code(f(S.BLS12_377, bytes(4 * u1), bytes(u1), None, bytes(2 * u1))) is S.InvalidArgument
    assert _code(f(6, bytes(4 * u1), bytes(u1), bytes(2 * u1), bytes(2 * u1))) is S.InvalidArgument
