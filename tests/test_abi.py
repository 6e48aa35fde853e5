"""The C-ABI library loads without a GPU, exports every symbol include/*.h declares, and its host-only
entry points (size arithmetic) agree with the reference's formulas; compute calls fail loudly (no CPU
fallback) when no device exists."""
import ctypes
import os
import re

import pytest

import pyref as R
import snark_setup_b200 as S
from snark_setup_b200 import ffi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZE_FIELDS = ("powers_length", "powers_g1_length", "g1_chunk_size", "other_chunk_size", "accumulator_size",
               "contribution_size", "public_key_size", "hash_size")


def _have_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "snark_setup_b200.h")).read()
    names = sorted(set(re.findall(r"^(?:int|void|size_t|const char\*)\s+(ss_[a-z0-9_]+)\s*\(", hdr, re.M)))
    assert len(names) >= 15
    L = ctypes.CDLL(S.lib_path)
    for n in names:
        assert hasattr(L, n), f"{n} declared in the header but not exported"


def test_sizes_match_reference_formulas():
    assert [S.element_size(S.BLS12_377, g, c) for g in (0, 1) for c in (0, 1)] == [96, 48, 192, 96]
    assert [S.element_size(S.BW6_761, g, c) for g in (0, 1) for c in (0, 1)] == [192, 96, 192, 96]
    assert (S.scalar_size(S.BLS12_377), S.scalar_size(S.BW6_761)) == (32, 48)
    for cid, cv in ((S.BLS12_377, R.BLS12_377), (S.BW6_761, R.BW6_761)):
        for k, bs, mode, ci, cs in ((10, 256, 0, 0, 0), (20, 256, 0, 0, 0), (4, 8, 1, 0, 8), (4, 8, 1, 1, 8), (4, 8, 1, 2, 8),
                                    (4, 8, 1, 3, 8), (5, 7, 1, 2, 20)):
            a = S.Phase1Parameters(cid, k, bs, mode, ci, cs)
            b = R.Phase1Parameters(cv, k, bs, mode, ci, cs)
            for f in SIZE_FIELDS:
                assert getattr(a, f) == getattr(b, f), (cv.name, k, mode, ci, f)
        # Marlin: tau_g1 over 2^k powers, plus k+2 tau_g2 and 3+3k alpha_g1 elements in the buffer of chunk 0 only
        for k, bs, mode, ci, cs in ((3, 8, 0, 0, 0), (3, 8, 1, 0, 4), (3, 8, 1, 1, 4), (4, 8, 1, 3, 4), (5, 7, 1, 2, 12),
                                    (10, 256, 0, 0, 0)):
            a = S.Phase1Parameters(cid, k, bs, mode, ci, cs, 1)
            b = R.Phase1Parameters(cv, k, bs, mode, ci, cs, R.MARLIN)
            for f in SIZE_FIELDS:
                assert getattr(a, f) == getattr(b, f), (cv.name, "marlin", k, mode, ci, f)
    with pytest.raises(ffi.InvalidChunk):  # a Marlin chunk must start below 2^power
        S.Phase1Parameters(S.BLS12_377, 3, 8, 1, 2, 4, 1)


def test_relayout_length_errors_without_device():
    """decompress / split / aggregation check their buffers against the layout before any device call."""
    full = S.Phase1Parameters(S.BLS12_377, 3, 8)
    chunk = S.Phase1Parameters(S.BLS12_377, 3, 8, 1, 1, 4)
    with pytest.raises(S.InvalidLength) as ei:  # compressed full accumulator
        S.phase1_decompress(full, bytes(100))
    assert (ei.value.expected, ei.value.got) == (2416, 100)
    with pytest.raises(S.InvalidLength) as ei:  # uncompressed full accumulator
        S.phase1_split_chunk(chunk, bytes(100), False, False)
    assert (ei.value.expected, ei.value.got) == (4768, 100)
    with pytest.raises(S.InvalidLength) as ei:  # compressed chunk 1 of size 4
        S.phase1_aggregate_chunk(chunk, bytes(10), True, bytearray(full.get_length(False)), False)
    assert (ei.value.expected, ei.value.got) == (1120, 10)


def test_argument_errors_are_reported_without_device():
    with pytest.raises(S.InvalidLength) as ei:
        S.batch_exp(S.BLS12_377, S.G1, bytearray(96 * 3), [1, 2])
    assert (ei.value.expected, ei.value.got) == (3, 2)
    with pytest.raises(S.SetupError):
        S.Phase1Parameters(7, 10, 256)


def test_prepare_phase2_and_qap_host_logic_without_device():
    """Sizes and argument validation of the SURVEY §8(f) entry points are host arithmetic (no compute call)."""
    # groth16_utils.rs:65-69,134-168: domain = next power of two; bytes of Groth16Params::write
    for cid, (u1, u2, c1, c2) in ((S.BLS12_377, (96, 192, 48, 96)), (S.BW6_761, (192, 192, 96, 96))):
        for size, m in ((1, 1), (2, 2), (3, 4), (1000, 1024), (1 << 20, 1 << 20), ((1 << 20) + 1, 1 << 21)):
            assert S.groth16_params_size(cid, size, False) == (m, 2 * u1 + u2 + 3 * m * u1 + m * u2 + (m - 1) * u1)
            assert S.groth16_params_size(cid, size, True) == (m, 2 * c1 + c2 + 3 * m * c1 + m * c2 + (m - 1) * c1)
    with pytest.raises(S.SetupError):          # 3 is not a radix-2 domain
        S.group_ifft(S.BLS12_377, S.G1, bytes(96 * 3), False, False)
    with pytest.raises(S.InvalidLength) as ei:  # h_query needs 2*degree - 1 powers (index panic in the reference)
        S.h_query_groth16(S.BLS12_377, bytes(96 * 6), False, 4, False)
    assert (ei.value.expected, ei.value.got) == (7, 6)
    sp = S.Phase1Parameters(S.BLS12_377, 3, 8)
    with pytest.raises(S.InvalidLength):        # domain 16 > 8 powers (groth16_utils.rs large_phase2_fails)
        S.groth16_params_new(sp, bytes(sp.get_length(False)), False, 9, False)
    with pytest.raises(S.InvalidLength):        # accumulator buffer too short
        S.groth16_params_new(sp, bytes(100), False, 8, False)
    bases = bytes(96 * 4)
    with pytest.raises(S.InvalidLength):        # coeffs[ind] out of range
        S.qap_dot_product(S.BLS12_377, S.G1, bases, False, [[(1, 4)]], False)
    with pytest.raises(S.InvalidData):          # scalar >= r
        S.qap_dot_product(S.BLS12_377, S.G1, bases, False, [[(R.BLS12_377.r, 0)]], False)


@pytest.mark.skipif(_have_gpu(), reason="box has a GPU")
def test_no_cpu_fallback():
    with pytest.raises(S.DeviceError):
        S.generate_powers_of_tau(S.BLS12_377, 5, 0, 4)
    with pytest.raises(S.DeviceError):
        S.apply_powers(S.BLS12_377, S.G1, bytes(96), False, S.CHECK_NO, True, 1, tau=3)
    g1, g2 = R.BLS12_377.g1, R.BLS12_377.g2
    with pytest.raises(S.DeviceError):
        S.group_ifft(S.BLS12_377, S.G1, g1.encode(g1.gen, False) * 4, False, False)
    with pytest.raises(S.DeviceError):
        S.same_ratio(S.BLS12_377, g1.encode(g1.gen, False) * 2, g2.encode(g2.gen, False) * 2)
    with pytest.raises(S.DeviceError):
        S.qap_dot_product(S.BLS12_377, S.G1, g1.encode(g1.gen, False) * 2, False, [[(1, 0)]], False)


def test_iter_chunk_matches_reference_schedule():
    """phase1/src/helpers/buffers.rs:22-73 against the oracle restatement, incl. the SURVEY A5 example."""
    for cid, cv in ((S.BLS12_377, R.BLS12_377),):
        for k, bs, mode, ci, cs in ((10, 256, 0, 0, 0), (3, 4, 0, 0, 0), (4, 5, 1, 0, 8), (4, 5, 1, 1, 8), (4, 5, 1, 3, 8),
                                    (4, 2, 0, 0, 0), (5, 7, 1, 2, 20), (4, 16, 1, 3, 8), (2, 64, 0, 0, 0)):
            a = S.Phase1Parameters(cid, k, bs, mode, ci, cs).iter_chunk()
            b = R.iter_chunk(R.Phase1Parameters(cv, k, bs, mode, ci, cs))
            assert a == b, (k, bs, mode, ci, cs)
    w = S.Phase1Parameters(S.BLS12_377, 10, 256).iter_chunk()
    assert len(w) == 9 and w[0] == (0, 256) and w[1] == (255, 511) and w[-1] == (2040, 2047)
