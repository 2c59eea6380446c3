"""K14 pin: the oracle's ObBitmap::get_row_ids restatement (and, on the GPU box, obgpu_bitmap_to_row_ids) against the REAL
common::ObBitmap (oracle/_ref/libref_bitmap.so, compiled from the reference's deps/oblib/src/lib/container/ob_bitmap.cpp when its
sources are present; otherwise the row ids it returned for tests/golden/ref_vectors.npz): window / limit / id_offset sweeps, `from`
advance, empty / full / sparse / dense bitmaps."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora


def _ref(required=True):
    """The live reference library; without it None, or a skip when the test checks nothing but the reference itself."""
    if not os.path.exists(ora.REF_BITMAP_LIB):
        if required:
            pytest.skip("oracle/_ref/libref_bitmap.so not built (needs the reference's sources)")
        return None
    L = C.CDLL(ora.REF_BITMAP_LIB)
    L.ref_bitmap_create.restype = C.c_void_p
    L.ref_bitmap_create.argtypes = [C.c_void_p, C.c_int64]
    L.ref_bitmap_destroy.argtypes = [C.c_void_p]
    L.ref_bitmap_get_row_ids.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int64, C.c_int64, C.c_int64]
    L.ref_bitmap_popcnt.restype = C.c_uint64
    L.ref_bitmap_popcnt.argtypes = [C.c_void_p]
    for f in ("ref_bitmap_and", "ref_bitmap_or"):
        getattr(L, f).argtypes = [C.c_void_p, C.c_void_p]
    L.ref_bitmap_not.argtypes = [C.c_void_p]
    L.ref_bitmap_bytes.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    L.ref_bitmap_next_valid_idx.restype = C.c_int64
    L.ref_bitmap_next_valid_idx.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int]
    return L


def ref_get_row_ids(L, bm, frm, to, limit, id_offset=0):
    h = L.ref_bitmap_create(bm.ctypes.data, bm.size)
    ids = np.zeros(max(limit, 1) + 8, dtype=np.int32)
    cnt, f = C.c_int64(0), C.c_int64(frm)
    ret = L.ref_bitmap_get_row_ids(h, ids.ctypes.data, C.byref(cnt), C.byref(f), to, limit, id_offset)
    L.ref_bitmap_destroy(h)
    return ret, ids[:cnt.value].copy(), f.value


def cases():
    rng = np.random.default_rng(17)
    for n in (1, 7, 64, 65, 200, 1000, 4099):
        for dens in (0.0, 0.02, 0.5, 0.97, 1.0):
            bm = (rng.random(n) < dens).astype(np.uint8)
            for _ in range(6):
                frm = int(rng.integers(0, n))
                to = int(rng.integers(frm, n + 1))
                limit = int(rng.choice([1, 2, 17, 256, 5000]))
                off = int(rng.integers(0, frm + 1))
                yield bm, frm, to, limit, off


def reference_row_ids(L):
    """(bitmap, from, to, limit, id_offset, the reference's row ids, its `from` after the call): from the live library L over
    cases(), or the committed golden answers when L is None."""
    if L is not None:
        for bm, frm, to, limit, off in cases():
            ret, want, wfrom = ref_get_row_ids(L, bm, frm, to, limit, off)
            assert ret == 0
            yield bm, frm, to, limit, off, want, wfrom
        return
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz"))
    for (bpos, n, frm, to, limit, off, ret, cnt, wfrom, ipos) in G["bitmap_cases"]:
        if ret == 0:
            yield (np.ascontiguousarray(G["bitmap_bytes"][bpos:bpos + n]), int(frm), int(to), int(limit), int(off),
                   G["bitmap_ids"][ipos:ipos + cnt], int(wfrom))


def test_oracle_get_row_ids_equals_the_reference():
    L = _ref(required=False)
    k = 0
    for bm, frm, to, limit, off, want, wfrom in reference_row_ids(L):
        got, gfrom = ora.bitmap_get_row_ids(bm, frm, to, limit, id_offset=off)
        assert np.array_equal(got, want) and gfrom == wfrom, (bm.size, frm, to, limit, off)
        k += 1
    assert k > (200 if L is not None else 50)


def test_logic_ops_and_popcnt_of_the_reference_are_bytewise():
    """bit_and / bit_or / bit_not / popcnt of the real ObBitmap == plain byte arithmetic on 0x00 / 0x01 images, which is what
    the oracle's filter-tree fold and the device's packed-word fold implement."""
    L = _ref()
    rng = np.random.default_rng(3)
    for n in (1, 63, 64, 1000, 1031):
        a = (rng.random(n) < 0.4).astype(np.uint8)
        b = (rng.random(n) < 0.6).astype(np.uint8)
        ha, hb = L.ref_bitmap_create(a.ctypes.data, n), L.ref_bitmap_create(b.ctypes.data, n)
        assert L.ref_bitmap_popcnt(ha) == int(a.sum())
        assert L.ref_bitmap_and(ha, hb) == 0
        out = np.zeros(n, dtype=np.uint8)
        L.ref_bitmap_bytes(ha, out.ctypes.data, n)
        assert np.array_equal(out, a & b)
        assert L.ref_bitmap_or(ha, hb) == 0
        L.ref_bitmap_bytes(ha, out.ctypes.data, n)
        assert np.array_equal(out, (a & b) | b)
        assert L.ref_bitmap_not(ha) == 0
        L.ref_bitmap_bytes(ha, out.ctypes.data, n)
        assert np.array_equal(out, 1 - ((a & b) | b))
        L.ref_bitmap_destroy(ha)
        L.ref_bitmap_destroy(hb)


@pytest.mark.gpu
def test_device_bitmap_to_row_ids_equals_the_reference():
    import oceanbase_b200 as ob
    ctx = ob.ScanContext(0)
    for i, (bm, frm, to, limit, off, want, wfrom) in enumerate(reference_row_ids(_ref(required=False))):
        if i % 3:
            continue
        got, gfrom = ctx.bitmap_to_row_ids(bm, frm, to, limit, id_offset=off)
        assert np.array_equal(got, want) and gfrom == wfrom, (bm.size, frm, to, limit, off)
    ctx.close()
