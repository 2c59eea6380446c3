"""Column checksums (K16): the oracle's restatement of ObMicroBlockChecksumHelper::cal_column_checksum
(blocksstable/ob_micro_block_checksum_helper.cpp:127-257) -- per cell ObDatum::checksum(0) (share/datum/ob_datum.h:849-856),
summed with int64 wrap-around -- pinned to the REAL reference's crc (oracle/_ref/libref_misc.so compiled from the reference's
ob_crc64_sse42 when its sources are present; otherwise the oracle's crc, which tests/test_checksum_ref_kat.py pins to the
reference's committed checksums) composed exactly as ob_datum.h composes it, and to the fixed points the sse4.2 loop of the
reference uses (null_pack_checksum / len_pack_checksum, :160-176)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora


def _ref_crc():
    """ob_crc64_sse42(seed, ptr, len) of the live reference library, or the oracle's when it could not be built."""
    if not os.path.exists(ora.REF_MISC_LIB):
        return ora.oracle().ora_crc64_sse42
    L = C.CDLL(ora.REF_MISC_LIB)
    L.ref_crc64_sse42.restype = C.c_uint64
    L.ref_crc64_sse42.argtypes = [C.c_uint64, C.c_void_p, C.c_int64]
    return L.ref_crc64_sse42


def ref_datum_checksum(crc, value: int, is_null: bool, datum_len: int) -> int:
    pack = np.array([0x80000000 if is_null else datum_len], dtype=np.uint32)
    c = crc(0, pack.ctypes.data, 4)
    if not is_null and datum_len > 0:
        v = np.array([value], dtype=np.int64)
        c = crc(c, v.ctypes.data, datum_len)
    return c


@pytest.mark.parametrize("datum_len", [8, 4, 1])
def test_oracle_column_checksum_is_the_sum_of_reference_datum_checksums(datum_len):
    crc = _ref_crc()
    o = ora.oracle()
    rng = np.random.default_rng(40 + datum_len)
    n = 3000
    vals = rng.integers(-2**62, 2**62, size=n, dtype=np.int64)
    if datum_len < 8:
        vals &= (1 << (8 * datum_len)) - 1
    nulls = (rng.random(n) < 0.2).astype(np.uint8)
    want = 0
    for r in range(n):
        want = (want + ref_datum_checksum(crc, int(vals[r]), bool(nulls[r]), datum_len)) & 0xffffffffffffffff
    want = want - (1 << 64) if want >= (1 << 63) else want
    assert o.ora_column_checksum(vals.ctypes.data, nulls.ctypes.data, n, datum_len) == want
    # no NULL array == no NULL cell
    want2 = 0
    for r in range(n):
        want2 = (want2 + ref_datum_checksum(crc, int(vals[r]), False, datum_len)) & 0xffffffffffffffff
    want2 = want2 - (1 << 64) if want2 >= (1 << 63) else want2
    assert o.ora_column_checksum(vals.ctypes.data, None, n, datum_len) == want2


def test_pack_fixed_points():
    """The sse4.2 loop hoists crc32(0, pack_) of a NULL datum and of a len-L datum out of the row loop; both are plain
    crc32c values of 4 little-endian bytes."""
    crc = _ref_crc()
    o = ora.oracle()
    one = np.zeros(1, dtype=np.int64)
    nl = np.ones(1, dtype=np.uint8)
    null_pack = np.array([0x80000000], dtype=np.uint32)
    assert o.ora_column_checksum(one.ctypes.data, nl.ctypes.data, 1, 8) == crc(0, null_pack.ctypes.data, 4)
    # 1000 NULL cells: 1000 x the same value
    many = np.zeros(1000, dtype=np.int64)
    nls = np.ones(1000, dtype=np.uint8)
    assert o.ora_column_checksum(many.ctypes.data, nls.ctypes.data, 1000, 8) == 1000 * crc(0, null_pack.ctypes.data, 4)
