"""Bit-stream primitives of the oracle pinned against (a) the reference's own known-answer tests
(unittest/storage/blocksstable/encoding/test_bit_stream.cpp:151-200) and (b) the REAL reference
ObBitStream compiled into oracle/_ref/libref_bitstream.so when the reference's sources are present, otherwise the
bytes its memory_safe_set wrote for tests/golden/ref_vectors.npz."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora


def _buf(n):
    return np.zeros(n, dtype=np.uint8)


def reference_bitstreams(R, widths, n, seed):
    """(width, values, the bytes the reference's memory_safe_set packs them into): from the live library R, or the committed
    golden streams (50 values per width) when R is None."""
    rng = np.random.default_rng(seed)
    if R is None:
        G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz"))
        index = {int(w): (int(pos), int(nbytes)) for (w, pos, nbytes) in G["bitstream_index"]}
        for width in widths:
            pos, nbytes = index[width]
            yield width, G["bitstream_values"][(width - 1) * 50:width * 50], np.ascontiguousarray(G["bitstream_bytes"][pos:pos + nbytes])
        return
    for width in widths:
        vals = rng.integers(0, 1 << 63, size=n, dtype=np.uint64)
        if width < 64:
            vals &= np.uint64((1 << width) - 1)
        a = _buf((n * width + 7) // 8 + 16)
        for i in range(n):
            R.ref_bs_memory_safe_set(a.ctypes.data, i * width, width, int(vals[i]))
        yield width, vals, a


def test_get_26_kat():
    # TEST(ObBitStream, get_26): 16 values x 13 bits written with memory_safe_set, read with the
    # PACKED_LEN_LESS_THAN_26 fast path
    L = ora.oracle()
    buf = _buf(64)
    cnt = 13
    for i in range(16):
        L.ora_bs_set(buf.ctypes.data, i * cnt, cnt, i)
    for i in range(16):
        assert L.ora_bs_get_fast(buf.ctypes.data, i * cnt, cnt, 32 * 8) == i
        assert L.ora_bs_get(buf.ctypes.data, i * cnt, cnt) == i


def test_perf_kat():
    # TEST(ObBitStream, perf): 25 values x 18 bits; generic get == fast get
    L = ora.oracle()
    buf = _buf(25 * 4 + 16)
    cnt = 18
    for i in range(25):
        L.ora_bs_set(buf.ctypes.data, i * cnt, cnt, i)
    for i in range(25):
        a = L.ora_bs_get(buf.ctypes.data, i * cnt, cnt)
        b = L.ora_bs_get_fast(buf.ctypes.data, i * cnt, cnt, 25 * 8 * 4)
        assert a == b == i


def test_set_get_random_widths():
    # TEST(ObBitStream, set_get): 100 random values with random widths 1..63, even then odd slots
    L = ora.oracle()
    rng = np.random.default_rng(20260922)
    data = rng.integers(0, 1 << 63, size=100, dtype=np.uint64)
    data[0] = 0
    bits = rng.integers(1, 64, size=100)
    total = int(bits.sum())
    buf = _buf(total // 8 + 16)
    off = np.concatenate([[0], np.cumsum(bits)[:-1]])
    for parity in (0, 1):
        for i in range(parity, 100, 2):
            L.ora_bs_set(buf.ctypes.data, int(off[i]), int(bits[i]), int(data[i]) & ((1 << int(bits[i])) - 1))
    for i in range(100):
        m = (1 << int(bits[i])) - 1
        assert L.ora_bs_get(buf.ctypes.data, int(off[i]), int(bits[i])) == int(data[i]) & m
    # negative integers (two's complement images)
    buf[:] = 0
    neg = (np.uint64(0) - data)
    for i in range(100):
        L.ora_bs_set(buf.ctypes.data, int(off[i]), int(bits[i]), int(neg[i]) & ((1 << int(bits[i])) - 1))
    for i in range(100):
        m = (1 << int(bits[i])) - 1
        assert L.ora_bs_get(buf.ctypes.data, int(off[i]), int(bits[i])) == int(neg[i]) & m


def test_oracle_matches_real_reference_bitstream():
    """Same random streams through the reference's ObBitStream and the oracle restatement:
    memory_safe_set / set produce identical bytes, get / get<unpack> return identical values."""
    L, R = ora.oracle(), ora.ref_bitstream()
    for width, vals, a in reference_bitstreams(R, range(1, 65), 257, 7):
        n, nbytes = len(vals), a.size
        b, c = _buf(nbytes), _buf(nbytes)
        for i in range(n):
            L.ora_bs_set(b.ctypes.data, i * width, width, int(vals[i]))
            if R is not None and width < 64:
                v = int(vals[i])
                assert R.ref_bs_set(c.ctypes.data, nbytes, i * width, width, v if v < (1 << 63) else v - (1 << 64)) == 0
        assert np.array_equal(a, b), f"width {width}: packed bytes differ from the reference"
        if R is not None and width < 64:
            assert np.array_equal(a, c)
        bs_len = n * width
        for i in range(n):
            want = int(vals[i])
            if R is not None:
                assert R.ref_bs_get(a.ctypes.data, i * width, width) == want
                assert R.ref_bs_get_unpack(a.ctypes.data, i * width, width, bs_len) == want
            assert L.ora_bs_get(a.ctypes.data, i * width, width) == want
            assert L.ora_bs_get_fast(a.ctypes.data, i * width, width, bs_len) == want
    if R is not None:
        for w in range(1, 65):
            assert R.ref_bs_get_mask(w) == (1 << w) - 1


def test_writer_bitpacking_matches_real_reference():
    """The host writer's packed RAW column bytes == what the reference's memory_safe_set emits."""
    import oceanbase_b200 as ob
    R = ora.ref_bitstream()
    packed = 0
    for width, vals, exp in reference_bitstreams(R, (1, 3, 7, 9, 13, 17, 21, 25, 26, 31, 33, 47, 57, 63), 300, 11):
        if R is not None:
            vals[0] = (1 << width) - 1  # force the width
            exp = _buf(exp.size)
            for i in range(len(vals)):
                R.ref_bs_memory_safe_set(exp.ctypes.data, i * width, width, int(vals[i]))
        n = len(vals)
        blk = ob.encode_block([ob.Column(ob.OBJ_UINT64, ob.ENC_RAW, vals.view(np.int64))])
        b = ora.Block(blk)
        hdr = blk[b.b.header_size:b.b.header_size + 16]
        attr, length = int(hdr[2]), int(hdr[12:16].view(np.uint32)[0])
        if not attr & 0x4:
            continue  # get_packing_size chose byte packing for this width
        assert length == width
        off = int(hdr[8:12].view(np.uint32)[0])
        meta = b.b.header_size + 16
        nbytes = (n * width + 7) // 8
        assert np.array_equal(blk[meta + off:meta + off + nbytes], exp[:nbytes])
        packed += 1
    assert packed > 0
