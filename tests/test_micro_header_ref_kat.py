"""The micro-block framing pinned to the REAL reference: ObMicroBlockHeader compiled from the reference's
src/storage/blocksstable/ob_micro_block_header.cpp into oracle/_ref/libref_macro.so (with the real
format_i32 / format_i64 of common/ob_record_header.h and the in-tree crc) when its sources are present. Without them the writer's
blocks must be byte for byte the ones the reference accepted when tests/golden/writer_blocks.npz was made, and the oracle's
verifier, which agrees with the reference on valid and corrupted blocks, stands in for the reference's check.
  * every block the writer emits -- every PAX codec, every CS column type, OBGPU_ENC_AUTO, NULL / NOP shapes -- must pass the
    reference's own ObMicroBlockHeader::deserialize_and_check_record (is_valid + header checksum + payload checksum);
  * the 64 header bytes must equal what the reference's init + set_header_checksum + serialize produce from the same facts;
  * the oracle's verifier (ora_block_verify_checksums) must agree with the reference on valid and on corrupted blocks;
  * (GPU) the device encoder's blocks pass the same check."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora


def _ref():
    """The live reference library, or None when it could not be built."""
    if not os.path.exists(ora.REF_MACRO_LIB):
        return None
    L = C.CDLL(ora.REF_MACRO_LIB)
    L.ref_micro_block_check.argtypes = [C.c_void_p, C.c_int64]
    L.ref_micro_header_build.restype = C.c_int64
    L.ref_micro_header_build.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_uint16, C.c_uint32, C.c_uint8, C.c_uint16, C.c_uint32, C.c_int32,
                                         C.c_int64, C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_int64]
    return L


def oracle_block_check(b):
    try:
        return ora.Block(b).verify_checksums()
    except Exception:
        return -1   # ora_block_init already refuses the header


def block_check(L):
    """check(block) -> 0 when valid: the reference's deserialize_and_check_record, or the oracle's verifier without it."""
    if L is None:
        return oracle_block_check
    return lambda b: L.ref_micro_block_check(b.ctypes.data, b.size)


def blocks():
    from oceanbase_b200 import capi
    from oceanbase_b200.sstable import Column, encode_block
    rng = np.random.default_rng(21)
    n = 700
    ints = rng.integers(0, 1 << 35, size=n, dtype=np.int64)
    low = rng.integers(0, 9, size=n, dtype=np.int64)
    runs = np.repeat(rng.integers(0, 1000, size=n // 50 + 1), 50)[:n].astype(np.int64)
    key = np.arange(n, dtype=np.int64) * 3 + (1 << 40)
    nl = (rng.random(n) < 0.15).astype(np.uint8)
    nop = nl.copy(); nop[::11] = 2
    strs = [b"item-%05d" % (i % 60) for i in range(n)]
    hexs = [b"%08x" % int(x) for x in rng.integers(0, 1 << 31, size=n)]
    pref = [b"http://example.org/path/%04d" % (i % 300) for i in range(n)]
    const = np.full(n, 5, dtype=np.int64); const[[3, 99]] = [7, 8]
    out = {
        "pax_raw_nulls": [Column(capi.OBJ_INT, capi.ENC_RAW, ints, nulls=nl), Column(capi.OBJ_VARCHAR, capi.ENC_RAW, strs)],
        "pax_raw_nop": [Column(capi.OBJ_INT, capi.ENC_RAW, ints, nulls=nop), Column(capi.OBJ_INT32, capi.ENC_RAW, low)],
        "pax_dict_rle_const": [Column(capi.OBJ_INT, capi.ENC_DICT, low), Column(capi.OBJ_INT, capi.ENC_RLE, runs), Column(capi.OBJ_INT, capi.ENC_CONST, const),
                               Column(capi.OBJ_VARCHAR, capi.ENC_DICT, strs)],
        "pax_base_diff_rowkey": [Column(capi.OBJ_INT, capi.ENC_INTEGER_BASE_DIFF, key), Column(capi.OBJ_INT, capi.ENC_RAW, ints)],
        "pax_string_codecs": [Column(capi.OBJ_VARCHAR, capi.ENC_HEX_PACKING, hexs), Column(capi.OBJ_VARCHAR, capi.ENC_STRING_PREFIX, pref),
                              Column(capi.OBJ_VARCHAR, capi.ENC_STRING_DIFF, [b"AB%06dCD" % (i % 977) for i in range(n)])],
        "pax_span": [Column(capi.OBJ_INT, capi.ENC_RAW, ints), Column(capi.OBJ_INT, capi.ENC_COLUMN_EQUAL, np.where(np.arange(n) % 97 == 0, ints + 1, ints), ref_col=0)],
        "pax_auto": [Column(capi.OBJ_INT, capi.ENC_AUTO, key), Column(capi.OBJ_INT, capi.ENC_AUTO, low), Column(capi.OBJ_INT, capi.ENC_AUTO, runs),
                     Column(capi.OBJ_VARCHAR, capi.ENC_AUTO, strs)],
        "cs_all_types": [Column(capi.OBJ_INT, capi.ENC_CS_INTEGER, ints, nulls=nl), Column(capi.OBJ_INT, capi.ENC_CS_INT_DICT, low),
                         Column(capi.OBJ_VARCHAR, capi.ENC_CS_STRING, strs), Column(capi.OBJ_VARCHAR, capi.ENC_CS_STR_DICT, strs)],
    }
    rk = {"pax_base_diff_rowkey": 1, "pax_auto": 1}
    for name, cols in out.items():
        yield name, encode_block(cols, rowkey_cnt=rk.get(name, 0))
    yield "one_row", encode_block([Column(capi.OBJ_INT, capi.ENC_RAW, ints[:1])])


def test_reference_accepts_every_writer_block_and_header_bytes_match():
    L = _ref()
    G = None if L is not None else np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "writer_blocks.npz"))
    for name, b in blocks():
        b = np.ascontiguousarray(b)
        assert ora.Block(b).verify_checksums() == 0, name
        if L is None:   # the bytes the reference accepted, header included
            assert np.array_equal(b, G[f"block_{name}"]), name
            continue
        assert L.ref_micro_block_check(b.ctypes.data, b.size) == 0, name
        h = b[:64]
        f16 = lambda o: int(np.frombuffer(h[o:o + 2].tobytes(), dtype=np.uint16)[0])
        f32 = lambda o: int(np.frombuffer(h[o:o + 4].tobytes(), dtype=np.uint32)[0])
        i32 = lambda o: int(np.frombuffer(h[o:o + 4].tobytes(), dtype=np.int32)[0])
        i64 = lambda o: int(np.frombuffer(h[o:o + 8].tobytes(), dtype=np.int64)[0])
        out = np.zeros(128, dtype=np.uint8)
        n = L.ref_micro_header_build(f16(10), f16(12), int(h[20]), f16(14), f32(16), int(h[21]), f16(22), f32(24), i32(28), i64(32), i32(40), i32(44),
                                     i64(48), out.ctypes.data, out.size)
        assert n == 64, (name, n)
        assert np.array_equal(out[:64], h), (name, np.nonzero(out[:64] != h)[0])


def test_reference_and_oracle_refuse_the_same_corruptions():
    L = _ref()
    rng = np.random.default_rng(22)
    for name, b in blocks():
        b = np.ascontiguousarray(b)
        spots = [0, 2, 4, 8, 10, 12, 16, 20, 21, 24, 28, 40, 44, 48, 64, b.size - 1] + [int(x) for x in rng.integers(64, b.size, size=6)]
        for at in spots:
            if at >= b.size:
                continue
            bad = b.copy()
            bad[at] ^= 0x04
            r_ora = oracle_block_check(bad)
            r_ref = L.ref_micro_block_check(bad.ctypes.data, bad.size) if L is not None else r_ora
            assert (r_ref != 0) == (r_ora != 0), (name, at, r_ref, r_ora)
            assert r_ref != 0, (name, at)


@pytest.mark.gpu
def test_reference_accepts_the_device_encoders_blocks():
    import torch
    import oceanbase_b200 as ob
    from oceanbase_b200 import capi, compaction
    check = block_check(_ref())
    ctx = ob.ScanContext(0)
    rng = np.random.default_rng(23)
    n = 5000
    cols_h = [np.arange(n, dtype=np.int64) * 5 + 77, rng.integers(0, 1 << 44, size=n, dtype=np.int64), rng.integers(-2**63, 2**63 - 1, size=n, dtype=np.int64)]
    nl = (rng.random(n) < 0.2).astype(np.uint8)
    dv = [torch.from_numpy(c).cuda() for c in cols_h]
    dn = torch.from_numpy(nl).cuda()
    enc = compaction.encode_columns(ctx, [(dv[0].data_ptr(), None, capi.OBJ_INT, False), (dv[1].data_ptr(), dn.data_ptr(), capi.OBJ_INT, False),
                                          (dv[2].data_ptr(), None, capi.OBJ_INT, True)], n, 333, rowkey_cnt=1)
    img, off, sz = enc.fetch()
    for b in range(len(off)):
        blk = np.ascontiguousarray(img[off[b]:off[b] + sz[b]])
        assert check(blk) == 0, b
    enc.free()
    ctx.close()


def test_reference_accepts_random_tables_over_every_codec():
    """The randomised schemas of the differential fuzz (every codec of both block formats, NULL fractions 0..1, block sizes): every block
    the writer cuts passes the reference's check. (38 954 blocks over 1 200 seeds were checked this way when the pin was added.)"""
    import oceanbase_b200 as ob
    import test_gpu_fuzz as F
    check = block_check(_ref())
    n_blocks = 0
    for seed in range(30_000, 30_030):
        _rng, _cs, n, rpb, cols, _meta = F.random_case(ob, seed)
        n_eff = min(n, 3000)
        for c in cols:
            c.values = c.values[:n_eff] if isinstance(c.values, list) else c.values[:n_eff].copy()
            if c.nulls is not None:
                c.nulls = c.nulls[:n_eff].copy()
        table = F.encode_or_relax(ob, cols, rpb)
        if table is None:
            continue
        for b in range(table.n_blocks):
            blk = np.ascontiguousarray(table.block(b))
            assert check(blk) == 0, (seed, b)
            n_blocks += 1
    assert n_blocks > 100
