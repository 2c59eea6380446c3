"""Two more building blocks pinned to the REAL reference (oracle/_ref/libref_misc.so, compiled from the reference's sources when
they are present; otherwise against the reference's answers committed in tests/golden/ref_vectors.npz):
  * ob_crc64_sse42 -- the micro-block payload checksum (ObMicroBlockHeader::data_checksum_, ob_micro_block_header.cpp:236-285)
    in the reference's three implementations (crc32 instruction, byte table, slicing-by-8; lib/checksum/ob_crc64.cpp:423-1103):
    the oracle's restatement, and the checksum the product's writer stores in every block header, must equal all three;
  * ObIntegerArray / ObIntArrayFuncTable lower_bound / upper_bound (encoding/ob_integer_array.h), the searches behind the RLE
    run lookup (ob_rle_decoder.cpp:25-49) and the CONST exception lookup (ob_const_decoder.cpp:93-121): the oracle's helpers,
    which its RLE / CONST decoders call, against them on every element width."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora


G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz"))


def _ref():
    """The live reference library, or None when it could not be built."""
    if not os.path.exists(ora.REF_MISC_LIB):
        return None
    L = C.CDLL(ora.REF_MISC_LIB)
    for f in ("ref_crc64_sse42", "ref_crc64_sse42_manually", "ref_fast_crc64_sse42_manually"):
        getattr(L, f).restype = C.c_uint64
        getattr(L, f).argtypes = [C.c_uint64, C.c_void_p, C.c_int64]
    L.ref_int_array_at.restype = C.c_int64
    L.ref_int_array_at.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    for f in ("ref_int_array_lower_bound", "ref_int_array_upper_bound"):
        getattr(L, f).restype = C.c_int64
        getattr(L, f).argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64]
    return L


def test_crc_known_answer():
    """crc32c("123456789") with seed 0 and no final xor is the complement-free form of the check value 0xE3069283:
    seed 0xffffffff then ^ 0xffffffff gives the standard one."""
    L = _ref()
    buf = np.frombuffer(b"123456789", dtype=np.uint8).copy()
    if L is not None:
        assert L.ref_crc64_sse42(0xffffffff, buf.ctypes.data, 9) ^ 0xffffffff == 0xE3069283
    assert ora.oracle().ora_crc64_sse42(0xffffffff, buf.ctypes.data, 9) ^ 0xffffffff == 0xE3069283


def test_oracle_crc_equals_all_three_reference_implementations():
    L = _ref()
    o = ora.oracle()
    if L is None:   # the reference's checksums of fixed buffers, lengths, alignments and seeds
        buf = np.ascontiguousarray(G["crc_buf"])
        for (n, shift, seed, want) in G["crc_cases"]:
            assert o.ora_crc64_sse42(int(seed), buf.ctypes.data + int(shift), int(n)) == int(want), (n, shift, seed)
        return
    rng = np.random.default_rng(20)
    big = rng.integers(0, 256, size=70_000, dtype=np.uint8)
    for n in list(range(0, 70)) + [127, 128, 129, 1000, 4095, 16384, 65537]:
        for shift in (0, 1, 3, 7):   # the hardware version first walks to an 8-byte boundary
            buf = big[shift:shift + n]
            p = big.ctypes.data + shift
            for seed in (0, 0x1234abcd, 0xffffffff):
                want = L.ref_crc64_sse42(seed, p, n)
                assert L.ref_crc64_sse42_manually(seed, p, n) == want
                assert L.ref_fast_crc64_sse42_manually(seed, p, n) == want
                assert o.ora_crc64_sse42(seed, p, n) == want, (n, shift, seed)
            del buf


def test_writer_block_checksums_against_the_reference():
    """data_checksum_ at header offset 48 covers the block after the header (data_zlength_ bytes, no compression)."""
    import oceanbase_b200 as ob
    L = _ref()
    rng = np.random.default_rng(4)
    n = 900
    strs = [bytes(rng.integers(97, 123, size=rng.integers(0, 20), dtype=np.uint8)) for _ in range(n)]
    for cols in ([ob.Column(ob.OBJ_INT, ob.ENC_RAW, rng.integers(-9, 9, size=n)), ob.Column(ob.OBJ_VARCHAR, ob.ENC_DICT, strs)],
                 [ob.Column(ob.OBJ_INT, ob.ENC_CS_INTEGER, rng.integers(0, 1 << 40, size=n)), ob.Column(ob.OBJ_VARCHAR, ob.ENC_CS_STRING, strs)]):
        blk = ob.encode_block(cols)
        b = ora.Block(blk)
        hs = b.b.header_size
        stored = int(blk[48:56].view(np.uint64)[0])
        zlen = int(blk[40:44].view(np.int32)[0])
        assert hs + zlen == len(blk)
        # without the reference: the oracle's crc, which test_oracle_crc_equals_all_three_reference_implementations pins to it
        crc = L.ref_crc64_sse42 if L is not None else ora.oracle().ora_crc64_sse42
        assert crc(0, blk.ctypes.data + hs, zlen) == stored
        assert b.verify_checksums() == 0


@pytest.mark.parametrize("byte", [1, 2, 4, 8])
def test_integer_array_searches(byte):
    L = _ref()
    o = ora.oracle()
    if L is None:   # the reference's lower / upper bounds over a fixed sorted array per width
        arr = np.ascontiguousarray(G[f"int_array_{byte}"])
        cases = G["int_array_cases"]
        cases = cases[cases[:, 0] == byte]
        assert len(cases) > 0
        for (_w, begin, end, k, lb, ub) in cases:
            assert o.ora_int_array_lower_bound(arr.ctypes.data, byte, int(begin), int(end), int(k)) == int(lb)
            assert o.ora_int_array_upper_bound(arr.ctypes.data, byte, int(begin), int(end), int(k)) == int(ub)
            assert lb == begin + int(np.searchsorted(arr[begin:end], k, side="left"))
            assert ub == begin + int(np.searchsorted(arr[begin:end], k, side="right"))
        return
    rng = np.random.default_rng(byte)
    dt = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}[byte]
    for n in (1, 2, 3, 17, 64, 255, 1000):
        hi = min((1 << (8 * byte)) - 1, 1 << 40)
        arr = np.sort(rng.integers(0, min(hi, 4 * n) + 1, size=n).astype(dt))   # duplicates on purpose
        keys = list(rng.integers(0, min(hi, 4 * n) + 1, size=40)) + [0, int(arr[0]), int(arr[-1]), int(arr[-1]) + 1 if int(arr[-1]) < hi else hi]
        for k in keys:
            k = int(k)
            for begin, end in ((0, n), (n // 3, n), (0, max(n // 2, 1))):
                lb = L.ref_int_array_lower_bound(arr.ctypes.data, byte, begin, end, k)
                ub = L.ref_int_array_upper_bound(arr.ctypes.data, byte, begin, end, k)
                assert o.ora_int_array_lower_bound(arr.ctypes.data, byte, begin, end, k) == lb
                assert o.ora_int_array_upper_bound(arr.ctypes.data, byte, begin, end, k) == ub
                assert lb == begin + int(np.searchsorted(arr[begin:end], k, side="left"))
                assert ub == begin + int(np.searchsorted(arr[begin:end], k, side="right"))
        for i in (0, n // 2, n - 1):
            assert L.ref_int_array_at(arr.ctypes.data, byte, i) == int(arr[i])
