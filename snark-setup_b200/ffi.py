"""ctypes binding of libsnarksetup_b200.so (include/snark_setup_b200.h).

Names, argument meaning and error behaviour follow the reference's Rust API so the parity tests read
like the reference's own tests (phase1/src/computation.rs:311-538, setup-utils/src/io/mod.rs:23-121).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
lib_path = os.environ.get("SS_LIB") or os.path.join(_CSRC, "libsnarksetup_b200.so")  # SS_LIB: A/B kernel variants

BLS12_377, BW6_761, MNT4_753, MNT6_753 = 0, 1, 2, 3
G1, G2 = 0, 1
CHECK_FULL, CHECK_ONLY_NON_ZERO, CHECK_ONLY_IN_GROUP, CHECK_NO = 0, 1, 2, 3
SUBGROUP_AUTO, SUBGROUP_DIRECT, SUBGROUP_BATCHED, SUBGROUP_NO = 0, 1, 2, 3
MODE_FULL, MODE_CHUNKED = 0, 1
GROTH16, MARLIN = 0, 1


class SetupError(Exception):
    """setup_utils::Error (setup-utils/src/errors.rs:11-38)."""

    def __init__(self, msg="", index=0, expected=0, got=0):
        super().__init__(msg)
        self.index, self.expected, self.got = index, expected, got


class InvalidData(SetupError): pass          # noqa: E701
class UnexpectedFlags(SetupError): pass      # noqa: E701
class PointAtInfinity(SetupError): pass      # noqa: E701
class IncorrectSubgroup(SetupError): pass    # noqa: E701
class InvalidLength(SetupError): pass        # noqa: E701
class InvalidChunk(SetupError): pass         # noqa: E701
class BatchTooSmall(SetupError): pass        # noqa: E701
class InvalidArgument(SetupError): pass      # noqa: E701
class DeviceError(SetupError): pass          # noqa: E701
class InvalidRatio(SetupError): pass         # noqa: E701  (VerificationError::InvalidRatio)


_ERRORS = {1: InvalidData, 2: UnexpectedFlags, 3: PointAtInfinity, 4: IncorrectSubgroup, 5: InvalidLength,
           6: InvalidChunk, 7: BatchTooSmall, 8: InvalidArgument, 9: DeviceError, 10: InvalidRatio}


class _ErrInfo(C.Structure):
    _fields_ = [("code", C.c_int), ("index", C.c_uint64), ("expected", C.c_uint64), ("got", C.c_uint64),
                ("message", C.c_char * 160)]


class _P1Params(C.Structure):
    _fields_ = [("curve", C.c_int), ("proving_system", C.c_int), ("contribution_mode", C.c_int),
                ("chunk_index", C.c_uint64), ("chunk_size", C.c_uint64), ("total_size_in_log2", C.c_uint32),
                ("batch_size", C.c_uint64)]


class _P1Sizes(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("powers_length", "powers_g1_length", "g1_chunk_size", "other_chunk_size",
                                          "accumulator_size", "contribution_size", "public_key_size", "hash_size")]


def build(verbose=False):
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-j8", "-C", _CSRC], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout[-4000:], r.stderr[-4000:])
    if r.returncode:
        raise RuntimeError("building libsnarksetup_b200.so failed")
    return lib_path


_lib = None


def lib():
    """The loaded CUDA library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(lib_path):
            raise DeviceError(f"{lib_path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'`; "
                              "there is no CPU fallback")
        L = C.CDLL(lib_path)
        L.ss_version.restype = C.c_char_p
        L.ss_element_size.restype = C.c_size_t
        L.ss_scalar_size.restype = C.c_size_t
        L.ss_last_error.argtypes = [C.POINTER(_ErrInfo)]
        L.ss_generate_powers_of_tau.argtypes = [C.c_int, C.c_char_p, C.c_uint64, C.c_uint64, C.c_void_p]
        L.ss_apply_powers.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_size_t,
                                      C.c_void_p, C.c_char_p, C.c_uint64, C.c_char_p]
        L.ss_batch_exp.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_char_p]
        L.ss_batch_mul.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_char_p]
        L.ss_transcode.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_size_t]
        L.ss_check_subgroup.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_int]
        L.ss_phase1_sizes_of.argtypes = [C.POINTER(_P1Params), C.POINTER(_P1Sizes)]
        L.ss_phase1_computation.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                            C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p]
        L.ss_phase1_computation_dev.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                                C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p,
                                                C.c_void_p]
        L.ss_init.argtypes = [C.POINTER(C.c_int), C.c_int]
        _lib = L
    return _lib


def _check(rc):
    if rc == 0:
        return
    info = _ErrInfo()
    lib().ss_last_error(C.byref(info))
    cls = _ERRORS.get(rc, SetupError)
    raise cls(info.message.decode(errors="replace"), info.index, info.expected, info.got)


class _ProfEntry(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("launches", C.c_uint64), ("elements", C.c_uint64), ("ms", C.c_double)]


def profile_enable(on=True):
    lib().ss_profile_enable(int(on))


def profile_reset():
    lib().ss_profile_reset()


def profile_launches():
    f = lib().ss_profile_launches
    f.restype = C.c_uint64
    return f()


def profile_read():
    """{kernel name: {"launches", "elements", "ms"}} accumulated since the last reset."""
    arr = (_ProfEntry * 64)()
    f = lib().ss_profile_read
    f.argtypes = [C.POINTER(_ProfEntry), C.c_int]
    n = f(arr, 64)
    return {arr[i].name.decode(): {"launches": arr[i].launches, "elements": arr[i].elements, "ms": arr[i].ms}
            for i in range(n)}


def set_concurrent_vectors(on=True):
    lib().ss_set_concurrent_vectors(int(on))


def init(devices=None):
    devices = list(devices or [])
    arr = (C.c_int * max(1, len(devices)))(*devices)
    _check(lib().ss_init(arr, len(devices)))


def element_size(curve, group, compressed):
    return lib().ss_element_size(curve, group, int(bool(compressed)))


def scalar_size(curve):
    return lib().ss_scalar_size(curve)


def _scalar(curve, v):
    if v is None:
        return None
    if isinstance(v, int):
        return v.to_bytes(scalar_size(curve), "little")
    return bytes(v)


def _buf(b):
    """(ctypes pointer, keepalive) for bytes / bytearray / memoryview / numpy arrays."""
    if isinstance(b, bytes):
        return C.cast(C.c_char_p(b), C.c_void_p), b
    if isinstance(b, bytearray):
        arr = (C.c_char * len(b)).from_buffer(b)
        return C.cast(arr, C.c_void_p), arr
    if hasattr(b, "ctypes"):  # numpy
        return C.c_void_p(b.ctypes.data), b
    mv = memoryview(b)
    arr = (C.c_char * mv.nbytes).from_buffer(mv)
    return C.cast(arr, C.c_void_p), arr


def generate_powers_of_tau(curve, tau, start, end):
    """setup-utils/src/helpers.rs:32-37 -> list of ints."""
    n = max(0, end - start)
    fb = scalar_size(curve)
    out = C.create_string_buffer(max(1, n * fb))
    _check(lib().ss_generate_powers_of_tau(curve, _scalar(curve, tau), start, end, out))
    return [int.from_bytes(out.raw[i * fb:(i + 1) * fb], "little") for i in range(n)]


def apply_powers(curve, group, inp, in_compressed, in_check, out_compressed, n, *, powers=None, tau=None,
                 first_power=0, coeff=None):
    """phase1/src/helpers/buffers.rs:77-97 on a slice that starts at element 0 of `inp`. Returns bytes."""
    fb = scalar_size(curve)
    osz = element_size(curve, group, out_compressed)
    out = bytearray(n * osz)
    pin, k1 = _buf(inp)
    pout, k2 = _buf(out) if n else (None, None)
    pw = None
    if powers is not None:
        pw = b"".join(int(p).to_bytes(fb, "little") for p in powers)
        if len(powers) != n:
            raise InvalidLength("powers", 0, n, len(powers))
    ppw, k3 = _buf(pw) if pw else (None, None)
    _check(lib().ss_apply_powers(curve, group, pin, int(in_compressed), in_check, pout, int(out_compressed), n, ppw,
                                 _scalar(curve, tau), first_power, _scalar(curve, coeff)))
    return bytes(out)


def batch_exp(curve, group, bases: bytearray, exps, coeff=None):
    """setup-utils/src/helpers.rs:75-140; `bases` = uncompressed elements, updated in place."""
    fb = scalar_size(curve)
    usz = element_size(curve, group, False)
    n = len(bases) // usz
    ex = b"".join(int(e).to_bytes(fb, "little") for e in exps)
    pb, k1 = _buf(bases) if n else (None, None)
    pe, k2 = _buf(ex) if ex else (None, None)
    _check(lib().ss_batch_exp(curve, group, pb, n, pe, len(exps), _scalar(curve, coeff)))


def batch_mul(curve, group, bases: bytearray, coeff):
    """setup-utils/src/helpers.rs:56-59."""
    usz = element_size(curve, group, False)
    n = len(bases) // usz
    pb, k1 = _buf(bases) if n else (None, None)
    _check(lib().ss_batch_mul(curve, group, pb, n, _scalar(curve, coeff)))


def transcode(curve, group, inp, in_compressed, check, out_compressed, n=None, want_output=True):
    """read_batch + write_batch (setup-utils/src/io/{read,write}.rs)."""
    isz = element_size(curve, group, in_compressed)
    osz = element_size(curve, group, out_compressed)
    if n is None:
        n = len(inp) // isz
    out = bytearray(n * osz) if want_output else None
    pin, k1 = _buf(inp) if n else (None, None)
    pout, k2 = _buf(out) if (want_output and n) else (None, None)
    _check(lib().ss_transcode(curve, group, pin, int(in_compressed), check, pout, int(out_compressed), n))
    return bytes(out) if want_output else None


def check_subgroup(curve, group, inp, compressed, mode=SUBGROUP_AUTO):
    """setup-utils/src/elements.rs:123-150."""
    sz = element_size(curve, group, compressed)
    n = len(inp) // sz
    pin, k1 = _buf(inp) if n else (None, None)
    _check(lib().ss_check_subgroup(curve, group, pin, int(compressed), n, mode))


def _rho_args(curve, rho, seed):
    fb = scalar_size(curve)
    prho = None
    keep = None
    if rho is not None:
        keep = b"".join(int(r).to_bytes(fb, "little") for r in rho)
        prho = C.cast(C.c_char_p(keep), C.c_void_p)
    pseed = bytes(seed) if seed is not None else None
    if pseed is not None and len(pseed) != 32:
        raise InvalidArgument("rho_seed must be 32 bytes")
    return prho, pseed, keep


def merge_pairs(curve, group, v1, v2, compressed, rho=None, seed=None, check=CHECK_NO):
    """setup-utils/src/helpers.rs:371-384 -> (s, sx) as uncompressed element bytes."""
    sz = element_size(curve, group, compressed)
    usz = element_size(curve, group, False)
    n = len(v1) // sz
    if len(v2) // sz != n:
        raise InvalidLength("merge_pairs", 0, n, len(v2) // sz)
    s, sx = C.create_string_buffer(usz), C.create_string_buffer(usz)
    p1, k1 = _buf(v1)
    p2, k2 = _buf(v2)
    prho, pseed, k3 = _rho_args(curve, rho, seed)
    f = lib().ss_merge_pairs
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_char_p,
                  C.c_void_p, C.c_void_p]
    _check(f(curve, group, p1, p2, int(compressed), check, n, prho, pseed, s, sx))
    return s.raw, sx.raw


def power_pairs(curve, group, v, compressed, rho=None, seed=None, check=CHECK_NO):
    """setup-utils/src/helpers.rs:388-390."""
    sz = element_size(curve, group, compressed)
    usz = element_size(curve, group, False)
    n = len(v) // sz
    s, sx = C.create_string_buffer(usz), C.create_string_buffer(usz)
    p1, k1 = _buf(v)
    prho, pseed, k3 = _rho_args(curve, rho, seed)
    f = lib().ss_power_pairs
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_char_p, C.c_void_p,
                  C.c_void_p]
    _check(f(curve, group, p1, int(compressed), check, n, prho, pseed, s, sx))
    return s.raw, sx.raw


def check_and_ratio(curve, group, inp, in_compressed, subgroup_mode=SUBGROUP_AUTO, do_ratio=True, rho=None, seed=None,
                    out_compressed=None):
    """accumulator.rs:95-145 + :56-91 + the re-emit of verification.rs:271-274 -> (out bytes | None, s, sx)."""
    sz = element_size(curve, group, in_compressed)
    usz = element_size(curve, group, False)
    n = len(inp) // sz
    s, sx = C.create_string_buffer(usz), C.create_string_buffer(usz)
    out = None
    pout = None
    if out_compressed is not None:
        out = bytearray(n * element_size(curve, group, out_compressed))
        pout, k0 = _buf(out) if n else (None, None)
    p1, k1 = _buf(inp) if n else (None, None)
    prho, pseed, k3 = _rho_args(curve, rho, seed)
    f = lib().ss_check_and_ratio
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_char_p,
                  C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    _check(f(curve, group, p1, int(in_compressed), n, subgroup_mode, int(do_ratio), prho, pseed, pout,
             int(bool(out_compressed)), s, sx))
    return (bytes(out) if out is not None else None), s.raw, sx.raw


def _split_pairs(curve, raw):
    u1, u2 = element_size(curve, G1, False), element_size(curve, G2, False)
    out, o = [], 0
    for usz in (u1, u2, u1, u1):
        out.append((raw[o:o + usz], raw[o + usz:o + 2 * usz]))
        o += 2 * usz
    return out


def pairs_size(curve):
    f = lib().ss_phase1_pairs_size
    f.restype = C.c_size_t
    return f(curve)


def phase1_verification_vectors(params, output, compressed_output, new_challenge, compressed_new_challenge,
                                subgroup_mode=SUBGROUP_AUTO, ratio_check=True, seed=None, shard=None, raw=False):
    """Hot loop of Phase1::verification (phase1/src/verification.rs:217-411).  `new_challenge` is a
    bytearray written in place (or None).  Returns [(s, sx)] for tau_g1, tau_g2, alpha_g1, beta_g1.
    shard=(index, count): only that index-range shard of every vector (partial sums; raw=True returns the blob
    ss_phase1_reduce_partial_pairs takes)."""
    cv = params.curve
    pairs = C.create_string_buffer(pairs_size(cv))
    pin, k1 = _buf(output)
    pnc, k2 = _buf(new_challenge) if new_challenge is not None else (None, None)
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase1_verification_vectors_shard
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                  C.c_int, C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]
    _check(f(C.byref(params.c), pin, len(output), int(compressed_output), pnc,
             len(new_challenge) if new_challenge is not None else 0, int(compressed_new_challenge), subgroup_mode,
             int(ratio_check), bytes(seed) if seed is not None else None, pairs, si, sc))
    return pairs.raw if raw else _split_pairs(cv, pairs.raw)


def phase1_verification_vectors_dev(params, d_output, output_len, compressed_output, d_new_challenge, nc_len,
                                    compressed_new_challenge, subgroup_mode=SUBGROUP_AUTO, ratio_check=True, seed=None,
                                    stream=0, shard=None, raw=False):
    cv = params.curve
    pairs = C.create_string_buffer(pairs_size(cv))
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase1_verification_vectors_shard_dev
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                  C.c_int, C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p]
    _check(f(C.byref(params.c), d_output, output_len, int(compressed_output), d_new_challenge, nc_len,
             int(compressed_new_challenge), subgroup_mode, int(ratio_check), bytes(seed) if seed is not None else None,
             pairs, si, sc, stream))
    return pairs.raw if raw else _split_pairs(cv, pairs.raw)


def phase1_reduce_partial_pairs(curve, blobs, raw=False):
    """Host-side reduction of the shards' partial (s, sx) (SURVEY.md §8e): element-wise group sums of the blobs."""
    n = pairs_size(curve)
    blobs = [bytes(b) for b in blobs]
    assert all(len(b) == n for b in blobs)
    out = C.create_string_buffer(n)
    f = lib().ss_phase1_reduce_partial_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_void_p]
    _check(f(curve, b"".join(blobs), len(blobs), out))
    return out.raw if raw else _split_pairs(curve, out.raw)


def set_strict_unchecked_inputs(on=True):
    lib().ss_set_strict_unchecked_inputs(1 if on else 0)


class Phase1Parameters:
    """phase1/src/objects/parameters.rs:115-294."""

    def __init__(self, curve, power, batch_size, mode=MODE_FULL, chunk_index=0, chunk_size=0, proving_system=GROTH16):
        self.c = _P1Params(curve, proving_system, mode, chunk_index, chunk_size, power, batch_size)
        z = _P1Sizes()
        _check(lib().ss_phase1_sizes_of(C.byref(self.c), C.byref(z)))
        for n, _ in _P1Sizes._fields_:
            setattr(self, n, getattr(z, n))
        self.curve = curve

    def get_length(self, compressed):
        return self.contribution_size - self.public_key_size if compressed else self.accumulator_size

    def iter_chunk(self):
        """phase1/src/helpers/buffers.rs:22-73 -> [(start, end)]."""
        f = lib().ss_phase1_iter_chunk
        f.argtypes = [C.POINTER(_P1Params), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_size_t, C.POINTER(C.c_size_t)]
        cnt = C.c_size_t(0)
        _check(f(C.byref(self.c), None, None, 0, C.byref(cnt)))
        a, b = (C.c_uint64 * max(1, cnt.value))(), (C.c_uint64 * max(1, cnt.value))()
        _check(f(C.byref(self.c), a, b, cnt.value, C.byref(cnt)))
        return [(a[i], b[i]) for i in range(cnt.value)]


def phase1_initialization(params, compressed_output):
    """Phase1::initialization (phase1/src/initialization.rs:12-57) -> the blank accumulator (hash prefix zero)."""
    f = lib().ss_phase1_initialization
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int]
    out = bytearray(params.get_length(compressed_output))
    po, k1 = _buf(out)
    _check(f(C.byref(params.c), po, len(out), int(compressed_output)))
    return bytes(out)


def phase1_aggregate_chunk(chunk_params, chunk, compressed_chunk, full: bytearray, compressed_full):
    """One iteration of Phase1::aggregation (phase1/src/aggregation.rs:11-180); `full` is written in place."""
    f = lib().ss_phase1_aggregate_chunk
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
    pc, k1 = _buf(chunk)
    pf, k2 = _buf(full)
    _check(f(C.byref(chunk_params.c), pc, len(chunk), int(compressed_chunk), pf, len(full), int(compressed_full)))


def phase1_split_chunk(chunk_params, full, compressed_full, compressed_chunk):
    """One iteration of Phase1::split (phase1/src/aggregation.rs:189-353) -> chunk bytes (hash prefix zero)."""
    f = lib().ss_phase1_split_chunk
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
    out = bytearray(chunk_params.get_length(compressed_chunk))
    pf, k1 = _buf(full)
    pc, k2 = _buf(out)
    _check(f(C.byref(chunk_params.c), pf, len(full), int(compressed_full), pc, len(out), int(compressed_chunk)))
    return bytes(out)


def phase1_decompress(params, inp, check=CHECK_NO):
    """helpers::accumulator::decompress (phase1/src/helpers/accumulator.rs:200-301)."""
    f = lib().ss_phase1_decompress
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_size_t]
    out = bytearray(params.get_length(False))
    pi, k1 = _buf(inp)
    po, k2 = _buf(out)
    _check(f(C.byref(params.c), pi, len(inp), check, po, len(out)))
    return bytes(out)


def group_ifft(curve, group, inp, in_compressed, out_compressed, check=CHECK_NO):
    """to_coeffs (setup-utils/src/groth16_utils.rs:44-53): group IFFT + normalize_batch -> bytes."""
    f = lib().ss_group_ifft
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_int]
    n = len(inp) // element_size(curve, group, in_compressed)
    out = bytearray(max(1, n) * element_size(curve, group, out_compressed))
    pi, k1 = _buf(inp)
    po, k2 = _buf(out)
    _check(f(curve, group, pi, int(in_compressed), check, n, po, int(out_compressed)))
    return bytes(out)


def h_query_groth16(curve, powers, in_compressed, degree, out_compressed, check=CHECK_NO):
    """h_query_groth16 (setup-utils/src/groth16_utils.rs:59-63) on serialized G1 powers -> bytes."""
    f = lib().ss_h_query_groth16
    f.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_size_t, C.c_void_p, C.c_int]
    n = len(powers) // element_size(curve, G1, in_compressed)
    out = bytearray(max(1, degree - 1) * element_size(curve, G1, out_compressed))
    pi, k1 = _buf(powers)
    po, k2 = _buf(out)
    _check(f(curve, pi, int(in_compressed), check, n, degree, po, int(out_compressed)))
    return bytes(out[:max(0, degree - 1) * element_size(curve, G1, out_compressed)])


def groth16_params_size(curve, phase2_size, compressed):
    """(domain_size, bytes written by Groth16Params::write) — setup-utils/src/groth16_utils.rs:65-69,134-168."""
    f = lib().ss_groth16_params_size
    f.argtypes = [C.c_int, C.c_uint64, C.c_int, C.POINTER(C.c_uint64), C.POINTER(C.c_size_t)]
    m, b = C.c_uint64(0), C.c_size_t(0)
    _check(f(curve, phase2_size, int(compressed), C.byref(m), C.byref(b)))
    return m.value, b.value


def groth16_params_new(params, accumulator, compressed_input, phase2_size, compressed_output, check=CHECK_NO):
    """Groth16Params::new + ::write (setup-utils/src/groth16_utils.rs:81-168) = prepare_phase2
    (phase2-cli/src/prepare_phase2.rs:16-70) -> the serialized parameters."""
    f = lib().ss_groth16_params_new
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint64, C.c_void_p, C.c_size_t,
                  C.c_int]
    _, nbytes = groth16_params_size(params.curve, phase2_size, compressed_output)
    out = bytearray(nbytes)
    pi, k1 = _buf(accumulator)
    po, k2 = _buf(out)
    _check(f(C.byref(params.c), pi, len(accumulator), int(compressed_input), check, phase2_size, po, len(out),
             int(compressed_output)))
    return bytes(out)


def same_ratio(curve, g1_pair, g2_pair):
    """setup-utils/src/helpers.rs:406-408; g1_pair / g2_pair = two uncompressed elements each -> bool."""
    f = lib().ss_same_ratio
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.POINTER(C.c_int)]
    same = C.c_int(0)
    _check(f(curve, bytes(g1_pair), bytes(g2_pair), C.byref(same)))
    return bool(same.value)


def check_same_ratio(curve, g1_pair, g2_pair):
    """setup-utils/src/helpers.rs:410-424; raises InvalidRatio."""
    f = lib().ss_check_same_ratio
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p]
    _check(f(curve, bytes(g1_pair), bytes(g2_pair)))


def check_same_ratio_batch(curve, g1_pairs, g2_pairs):
    """Several check_same_ratio in one launch; raises InvalidRatio with .index = first failing check."""
    f = lib().ss_check_same_ratio_batch
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_int, C.POINTER(C.c_int)]
    n = len(g1_pairs) // (2 * element_size(curve, G1, False))
    bad = C.c_int(-1)
    _check(f(curve, bytes(g1_pairs), bytes(g2_pairs), n, C.byref(bad)))


def phase1_check_ratio_pairs(curve, pairs, g1_check, g2_check):
    """The four check_same_ratio of a response from its (reduced) `pairs` blob; raises InvalidRatio (.index = vector)."""
    f = lib().ss_phase1_check_ratio_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_char_p]
    _check(f(curve, bytes(pairs), bytes(g1_check), bytes(g2_check)))


def phase1_verification_ratios(params, output, compressed_output, new_challenge, compressed_new_challenge,
                               check_output=CHECK_FULL, subgroup_mode=SUBGROUP_AUTO, seed=None):
    """Per-vector half of Phase1::verification with its verdict (phase1/src/verification.rs:44-80,217-411):
    raises PointAtInfinity / IncorrectSubgroup / InvalidRatio (.index = vector)."""
    f = lib().ss_phase1_verification_ratios
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.c_int,
                  C.c_int, C.c_char_p]
    pin, k1 = _buf(output)
    pnc, k2 = _buf(new_challenge) if new_challenge is not None else (None, None)
    _check(f(C.byref(params.c), pin, len(output), int(compressed_output), check_output, pnc,
             len(new_challenge) if new_challenge is not None else 0, int(compressed_new_challenge), subgroup_mode,
             bytes(seed) if seed is not None else None))


def qap_dot_product(curve, group, bases, bases_compressed, rows, out_compressed, check=CHECK_NO):
    """dot_product_vec + normalize_batch (phase2/src/polynomial.rs:30-47,75-94).  `rows` = per-variable lists
    [(coeff, index), ...] as MPCParameters::process_matrix builds them (phase2/src/parameters.rs:96-105)."""
    import array
    f = lib().ss_qap_dot_product
    f.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                  C.c_size_t, C.c_void_p, C.c_int]
    fb = scalar_size(curve)
    n = len(bases) // element_size(curve, group, bases_compressed)
    row_ptr = array.array("Q", [0])
    index = array.array("I")
    coeffs = bytearray()
    for row in rows:
        for c, i in row:
            index.append(i)
            coeffs += int(c).to_bytes(fb, "little")
        row_ptr.append(len(index))
    out = bytearray(max(1, len(rows)) * element_size(curve, group, out_compressed))
    pb, k1 = _buf(bases) if n else (None, None)
    po, k2 = _buf(out)
    prp, k3 = _buf(bytearray(row_ptr.tobytes()))
    pix, k4 = _buf(bytearray(index.tobytes())) if len(index) else (None, None)
    pco, k5 = _buf(coeffs) if len(coeffs) else (None, None)
    _check(f(curve, group, pb, int(bases_compressed), check, n, prp, pix, pco, len(rows), po, int(out_compressed)))
    return bytes(out[:len(rows) * element_size(curve, group, out_compressed)])


def phase1_computation(params: Phase1Parameters, inp, out, compressed_input, compressed_output, check_input,
                       tau, alpha, beta, shard=None):
    """Phase1::computation (phase1/src/computation.rs:16-308) on host buffers; `out` is written in place.
    shard=(index, count): only that index-range shard of every vector is read and written."""
    pin, k1 = _buf(inp)
    pout, k2 = _buf(out)
    cv = params.curve
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase1_computation_shard
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int,
                  C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32]
    _check(f(C.byref(params.c), pin, len(inp), pout, len(out), int(compressed_input), int(compressed_output),
             check_input, _scalar(cv, tau), _scalar(cv, alpha), _scalar(cv, beta), si, sc))


def phase1_computation_dev(params: Phase1Parameters, d_in, in_len, d_out, out_len, compressed_input,
                           compressed_output, check_input, tau, alpha, beta, stream=0, shard=None):
    """Same, on device pointers (ints) of the current CUDA device."""
    cv = params.curve
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase1_computation_shard_dev
    f.argtypes = [C.POINTER(_P1Params), C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int,
                  C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p]
    _check(f(C.byref(params.c), d_in, in_len, d_out, out_len, int(compressed_input), int(compressed_output),
             check_input, _scalar(cv, tau), _scalar(cv, alpha), _scalar(cv, beta), si, sc, stream))


# ---- phase 2: MPCParameters::contribute / verify on the H and L queries -----------------------------------------------
def phase2_pairs_size(curve):
    f = lib().ss_phase2_pairs_size
    f.restype = C.c_size_t
    return f(curve)


def _split_phase2_pairs(curve, raw):
    u = element_size(curve, G1, False)
    return [(raw[0:u], raw[u:2 * u]), (raw[2 * u:3 * u], raw[3 * u:4 * u])]


def phase2_contribute(curve, delta, h_query: bytearray, l_query: bytearray, compressed, check=CHECK_NO, delta_g1=None,
                      delta_g2=None, shard=None):
    """The hot half of MPCParameters::contribute (phase2/src/parameters.rs:286-307): h_query / l_query <- delta^-1 * each
    element and delta_g1 / delta_g2 <- delta * element, all serialized with `compressed` and updated IN PLACE
    (bytearrays; delta_g1 / delta_g2 may be None).  shard=(index, count): only that index-range shard of each query."""
    sz = element_size(curve, G1, compressed)
    nh, nl = len(h_query) // sz, len(l_query) // sz
    ph, k1 = _buf(h_query) if nh else (None, None)
    pl, k2 = _buf(l_query) if nl else (None, None)
    pd1, k3 = _buf(delta_g1) if delta_g1 is not None else (None, None)
    pd2, k4 = _buf(delta_g2) if delta_g2 is not None else (None, None)
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase2_contribute_shard
    f.argtypes = [C.c_int, C.c_char_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p,
                  C.c_void_p, C.c_uint32, C.c_uint32]
    _check(f(curve, _scalar(curve, delta), ph, nh, pl, nl, int(bool(compressed)), check, pd1, pd2, si, sc))


def phase2_verification_pairs(curve, h_before, h_after, l_before, l_after, compressed, check_before=CHECK_NO,
                              check_after=CHECK_ONLY_NON_ZERO, subgroup_mode=SUBGROUP_AUTO, seed=None, shard=None,
                              raw=False):
    """merge_pairs(before, after) of the H and L queries (phase2/src/parameters.rs:393-407) ->
    [(s_h, sx_h), (s_l, sx_l)] uncompressed, or the raw blob; shard=(index, count) gives that shard's partial sums."""
    sz = element_size(curve, G1, compressed)
    nh, nl = len(h_before) // sz, len(l_before) // sz
    if len(h_after) // sz != nh or len(l_after) // sz != nl:
        raise InvalidLength("before / after lengths differ", 0, nh, len(h_after) // sz)
    pairs = C.create_string_buffer(phase2_pairs_size(curve))
    bufs = [_buf(b) if len(b) else (None, None) for b in (h_before, h_after, l_before, l_after)]
    si, sc = shard if shard is not None else (0, 1)
    f = lib().ss_phase2_verification_pairs
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                  C.c_int, C.c_int, C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]
    _check(f(curve, bufs[0][0], bufs[1][0], nh, bufs[2][0], bufs[3][0], nl, int(bool(compressed)), check_before,
             check_after, subgroup_mode, bytes(seed) if seed is not None else None, pairs, si, sc))
    return pairs.raw if raw else _split_phase2_pairs(curve, pairs.raw)


def phase2_reduce_partial_pairs(curve, blobs, raw=False):
    """Element-wise group sums of the shards' partial phase-2 pairs blobs."""
    n = phase2_pairs_size(curve)
    blobs = [bytes(b) for b in blobs]
    assert all(len(b) == n for b in blobs)
    out = C.create_string_buffer(n)
    f = lib().ss_phase2_reduce_partial_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_void_p]
    _check(f(curve, b"".join(blobs), len(blobs), out))
    return out.raw if raw else _split_phase2_pairs(curve, out.raw)


def phase2_check_ratio_pairs(curve, pairs, delta_g1_after, delta_g2_before, delta_g2_after):
    """The three ratio checks of MPCParameters::verify from a pairs blob and uncompressed delta elements; raises
    InvalidRatio with .index 0 (delta), 1 (H) or 2 (L)."""
    f = lib().ss_phase2_check_ratio_pairs
    f.argtypes = [C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
    _check(f(curve, bytes(pairs), bytes(delta_g1_after), bytes(delta_g2_before), bytes(delta_g2_after)))


def phase2_verification(curve, h_before, h_after, l_before, l_after, compressed, delta_g1_after, delta_g2_before,
                        delta_g2_after, check_before=CHECK_NO, check_after=CHECK_ONLY_NON_ZERO,
                        subgroup_mode=SUBGROUP_AUTO, seed=None):
    """phase2_verification_pairs over the whole queries + phase2_check_ratio_pairs; the delta elements are serialized
    with `compressed`."""
    sz = element_size(curve, G1, compressed)
    nh, nl = len(h_before) // sz, len(l_before) // sz
    if len(h_after) // sz != nh or len(l_after) // sz != nl:
        raise InvalidLength("before / after lengths differ", 0, nh, len(h_after) // sz)
    bufs = [_buf(b) if len(b) else (None, None) for b in (h_before, h_after, l_before, l_after)]
    f = lib().ss_phase2_verification
    f.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_int,
                  C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
    _check(f(curve, bufs[0][0], bufs[1][0], nh, bufs[2][0], bufs[3][0], nl, int(bool(compressed)), check_before,
             check_after, subgroup_mode, bytes(delta_g1_after), bytes(delta_g2_before), bytes(delta_g2_after),
             bytes(seed) if seed is not None else None))
