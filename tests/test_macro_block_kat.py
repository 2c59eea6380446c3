"""Macro-block framing pinned to the REAL reference (oracle/_ref/libref_macro.so: ObMacroBlockCommonHeader and
ObSSTableMacroBlockHeader compiled from the reference's src/storage/blocksstable, with ob_crc64 for the payload checksum, when
its sources are present; without them the oracle's parser, which agrees with the reference's deserialize, reads the headers):
  * the headers the writer emits (obgpu_writer_build_macro_blocks) must be the bytes the reference's own init / serialize produce
    for the same facts, and the reference's deserialize + is_valid must accept them and read the same fields back;
  * the oracle's parser (ora_macro_block_parse / ora_macro_block_micro_blocks) must agree with the reference's deserialize and
    find exactly the micro-blocks the writer packed (bytes equal, checksums chained as ob_macro_block.cpp:301-303 does)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora

REF_MACRO_LIB = ora.REF_MACRO_LIB


def _ref(required=True):
    """The live reference library; without it None, or a skip when the test checks nothing but the reference itself."""
    if not os.path.exists(REF_MACRO_LIB):
        if required:
            pytest.skip("oracle/_ref/libref_macro.so not built (needs the reference's sources)")
        return None
    L = C.CDLL(REF_MACRO_LIB)
    L.ref_ob_crc64.restype = C.c_uint64
    L.ref_ob_crc64.argtypes = [C.c_void_p, C.c_int64]
    L.ref_macro_common_header_size.restype = C.c_int64
    L.ref_macro_fixed_header_size.restype = C.c_int64
    L.ref_macro_headers_build.restype = C.c_int64
    L.ref_macro_headers_build.argtypes = [C.c_uint16, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                          C.c_void_p, C.c_int64]
    L.ref_macro_headers_parse.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
    return L


def _oracle():
    O = ora.oracle()
    O.ora_macro_block_parse.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32]
    O.ora_macro_block_micro_blocks.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.c_int32]
    return O


def make_table(seed=1, n=60_000, rpb=700):
    from oceanbase_b200 import capi
    from oceanbase_b200.sstable import Column, encode_table
    rng = np.random.default_rng(seed)
    key = np.arange(n, dtype=np.int64) * 3 + 11
    cols = [Column(capi.OBJ_INT, capi.ENC_INTEGER_BASE_DIFF, key),
            Column(capi.OBJ_INT, capi.ENC_RAW, rng.integers(0, 1 << 40, size=n, dtype=np.int64), nulls=(rng.random(n) < 0.1).astype(np.uint8)),
            Column(capi.OBJ_INT32, capi.ENC_DICT, rng.integers(0, 50, size=n, dtype=np.int64)),
            Column(capi.OBJ_VARCHAR, capi.ENC_DICT, [b"v%03d" % (i % 37) for i in range(n)])]
    types = [capi.OBJ_INT, capi.OBJ_INT, capi.OBJ_INT32, capi.OBJ_VARCHAR]
    return encode_table(cols, rpb, rowkey_cnt=1), types


def test_struct_sizes():
    L = _ref()
    assert L.ref_macro_common_header_size() == 24
    assert L.ref_macro_fixed_header_size() == 128


@pytest.mark.parametrize("version,is_cg,macro_size,rows", [(1, False, 2 << 20, 400_000), (2, False, 256 << 10, 60_000), (1, True, 64 << 10, 60_000)])
def test_writer_headers_are_the_reference_bytes_and_parse_back(version, is_cg, macro_size, rows):
    from oceanbase_b200.sstable import build_macro_blocks
    L, O = _ref(required=False), _oracle()
    table, types = make_table(n=rows)
    orders = [0, -1, 0, 0]
    mi = build_macro_blocks(table, types, 1, tablet_id=200001, logical_version=7, first_data_seq=40, header_version=version, is_cg=is_cg,
                            macro_block_size=macro_size, col_orders=orders)
    assert mi.n_macro >= 2 and mi.first_micro[0] == 0 and mi.first_micro[-1] == table.n_blocks
    metas = np.zeros((4, 4), dtype=np.uint8)
    metas[:, 0] = types
    ords = np.array(orders, dtype=np.int32)
    for m in range(mi.n_macro):
        blk = np.ascontiguousarray(mi.image[m * macro_size:(m + 1) * macro_size])
        # ---- the reference parses the writer's block ------------------------------------------------------------------
        rf = np.zeros(28, dtype=np.int64)
        if L is not None:
            assert L.ref_macro_headers_parse(blk.ctypes.data, blk.size, rf.ctypes.data) == 0
        else:   # the oracle's parse, payload checksum checked
            assert O.ora_macro_block_parse(blk.ctypes.data, blk.size, rf.ctypes.data, 1) == 0
        lo, hi = int(mi.first_micro[m]), int(mi.first_micro[m + 1])
        want_rows = 0
        for b in range(lo, hi):
            want_rows += int(np.frombuffer(table.block(b)[16:20].tobytes(), dtype=np.uint32)[0])
        assert rf[17] == hi - lo and rf[15] == want_rows and rf[11] == 40 + m and rf[9] == 200001 and rf[10] == 7
        assert rf[12] == 4 and rf[13] == 1 and rf[7] == version and rf[26] == (1 if is_cg else 0) and rf[25] == 1
        assert rf[19] == int(table.sizes[lo:hi].sum()) and rf[16] == rf[18] + rf[19] and rf[4] == rf[16] - 24
        if L is not None:
            # payload checksum = (int32) ob_crc64(payload)
            pc = L.ref_ob_crc64(blk.ctypes.data + 24, int(rf[4]))
            assert np.int32(np.uint32(pc & 0xffffffff)) == np.int32(rf[5])
            # ---- the reference BUILDS the same headers from the same facts: byte equality --------------------------------
            out = np.zeros(4096, dtype=np.uint8)
            n = L.ref_macro_headers_build(version, 200001, 7, 40 + m, 4, 1, int(rf[14]), int(rf[15]), int(rf[17]), int(rf[19]), int(rf[16]),
                                          int(rf[24]), 1 if is_cg else 0, metas.ctypes.data, ords.ctypes.data, None, int(rf[4]),
                                          int(np.int32(rf[5])), out.ctypes.data, out.size)
            assert n == rf[18], (n, rf[18])
            got, want = blk[:n].copy(), out[:n].copy()
            got[24 + 121:24 + 128] = 0    # tail padding of FixedHeader (after encrypt_key_): not data
            want[24 + 121:24 + 128] = 0
            assert np.array_equal(got, want), np.nonzero(got != want)[0][:10]
        # ---- the oracle's parser agrees with the reference's deserialize and finds the packed micro-blocks ----------------
        of = np.zeros(28, dtype=np.int64)
        assert O.ora_macro_block_parse(blk.ctypes.data, blk.size, of.ctypes.data, 1) == 0
        assert np.array_equal(of, rf), (of, rf)
        offs, szs, cnt = np.zeros(hi - lo, dtype=np.int64), np.zeros(hi - lo, dtype=np.int64), C.c_int32(0)
        assert O.ora_macro_block_micro_blocks(blk.ctypes.data, blk.size, offs.ctypes.data, szs.ctypes.data, hi - lo, C.byref(cnt), 1) == 0
        assert cnt.value == hi - lo
        for i, b in enumerate(range(lo, hi)):
            assert szs[i] == table.sizes[b]
            assert np.array_equal(blk[offs[i]:offs[i] + szs[i]], table.block(b))


def test_corruption_is_refused_by_reference_and_oracle_alike():
    from oceanbase_b200.sstable import build_macro_blocks
    L, O = _ref(required=False), _oracle()
    table, types = make_table(seed=2, n=20_000)
    mi = build_macro_blocks(table, types, 1, macro_block_size=256 << 10)
    blk = np.ascontiguousarray(mi.image[:256 << 10]).copy()
    rf, of = np.zeros(28, dtype=np.int64), np.zeros(28, dtype=np.int64)
    for at, val in ((8, 77), (4, 9), (24 + 6, 1), (24 + 8, 0), (24 + 52, 0)):   # common magic, version; macro magic; tablet id 0; micro count 0
        bad = blk.copy()
        bad[at:at + 8 if at == 24 + 8 else at + (4 if at in (8, 4, 24 + 52) else 2)] = 0
        bad[at] = val
        r2 = O.ora_macro_block_parse(bad.ctypes.data, bad.size, of.ctypes.data, 0)
        r1 = L.ref_macro_headers_parse(bad.ctypes.data, bad.size, rf.ctypes.data) if L is not None else r2
        assert r1 != 0 and r2 != 0, (at, r1, r2)
    # a flipped payload byte: headers still parse, the checksum check refuses
    bad = blk.copy()
    bad[5000] ^= 0x40
    assert O.ora_macro_block_parse(bad.ctypes.data, bad.size, of.ctypes.data, 0) == 0
    assert O.ora_macro_block_parse(bad.ctypes.data, bad.size, of.ctypes.data, 1) != 0
