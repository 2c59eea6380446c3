"""K13 pin: the oracle's integer stream decoders (oracle/ob_stream_codecs.c) against the REAL reference codec library
(oracle/_ref/libref_codec.so, compiled by oracle/Makefile from the reference's deps/oblib/src/lib/codec when its sources are present).

Every codec x width decodes what the reference ENCODER produced and must equal both the input and the reference
DECODER's output. Datasets follow unittest/storage/blocksstable/cs_encoding/test_integer_stream.cpp:459-829
(all zero, min / max, monotone, negative deltas, long runs, random) plus exception-heavy PFOR blocks. Without the reference's
sources the same checks run on the streams the reference encoder produced for tests/golden/ref_vectors.npz."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_binding as ora

TYPES = {1: "RAW", 2: "DOUBLE_DELTA_ZIGZAG_RLE", 3: "DOUBLE_DELTA_ZIGZAG_PFOR", 4: "DELTA_ZIGZAG_RLE", 5: "DELTA_ZIGZAG_PFOR",
         6: "SIMD_FIXEDPFOR", 8: "XOR_FIXED_PFOR"}
WIDTHS = {1: np.uint8, 2: np.uint16, 4: np.uint32, 8: np.uint64}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz")


def datasets(dt, rng):
    bits = np.dtype(dt).itemsize * 8
    top = (1 << bits) - 1
    out = []
    for n in (1, 2, 5, 31, 127, 128, 129, 255, 256, 300, 1000, 2051):
        out.append(("zeros", np.zeros(n, dtype=dt)))
        out.append(("max", np.full(n, top, dtype=dt)))
        out.append(("minmax", np.array([0, top] * n, dtype=dt)[:n]))
        out.append(("mono", (np.arange(n, dtype=np.uint64) * 3 + 7).astype(dt)))
        out.append(("mono_desc", (np.uint64(top) - np.arange(n, dtype=np.uint64) * 5).astype(dt)))
        out.append(("runs", np.repeat(rng.integers(0, min(top, 1000) + 1, size=n // 40 + 1), 40)[:n].astype(dt)))
        out.append(("long_run_then_step", np.concatenate([np.full(n // 2 + 1, 9), np.full(n, 200 if top >= 200 else 3)])[:n].astype(dt)))
        out.append(("random_full", rng.integers(0, top, size=n, dtype=np.uint64, endpoint=True).astype(dt)))
        out.append(("random_small", rng.integers(0, 50, size=n).astype(dt)))
        spikes = rng.integers(0, 16, size=n).astype(np.uint64)
        spikes[rng.random(n) < 0.07] = top                    # PFOR exceptions
        out.append(("spikes", spikes.astype(dt)))
        walk = np.cumsum(rng.integers(-40, 41, size=n)).astype(np.int64) + (1 << (bits - 2))
        out.append(("walk", (walk.astype(np.uint64) & np.uint64(top)).astype(dt)))
        lin = (np.arange(n, dtype=np.uint64) * 1000 + 12345) & np.uint64(top)   # constant delta: double-delta runs
        out.append(("linear", lin.astype(dt)))
    return out


def _ref():
    """The live reference codec library, or None when it could not be built."""
    if not os.path.exists(ora.REF_CODEC_LIB):
        return None
    L = C.CDLL(ora.REF_CODEC_LIB)
    L.ref_codec_encode.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.POINTER(C.c_uint64)]
    L.ref_codec_decode.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.POINTER(C.c_uint64)]
    return L


def ref_encode(L, t, a):
    ub = a.dtype.itemsize
    out = np.zeros(a.size * ub * 2 + 4096, dtype=np.uint8)
    ol = C.c_uint64(0)
    r = L.ref_codec_encode(t, ub, a.ctypes.data, a.size, out.ctypes.data, out.size, C.byref(ol))
    assert r == 0, (t, ub, a.size, r)
    return out[:ol.value].copy()


def reference_streams(L, t, ub, seed):
    """(dataset name, values, the reference encoder's bytes) of codec t at width ub: from the live library L, or the committed
    golden streams when L is None."""
    dt = WIDTHS[ub]
    if L is not None:
        for name, a in datasets(dt, np.random.default_rng(seed)):
            a = np.ascontiguousarray(a)
            yield name, a, ref_encode(L, t, a)
        return
    G = np.load(GOLDEN)
    n_cases = 0
    for (gt, gub, n, vpos, epos, elen) in G["codec_index"]:
        if gt == t and gub == ub:
            n_cases += 1
            yield f"golden {n_cases}", G["codec_values"][vpos:vpos + n].astype(dt), G["codec_bytes"][epos:epos + elen]
    assert n_cases > 0, (t, ub)


@pytest.mark.parametrize("t", sorted(TYPES))
@pytest.mark.parametrize("ub", sorted(WIDTHS))
def test_oracle_decodes_reference_streams(t, ub):
    L = _ref()
    O = ora.oracle()
    O.ora_int_stream_decode.argtypes = [C.c_int32, C.c_uint32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.POINTER(C.c_int64)]
    dt = WIDTHS[ub]
    for name, a, enc in reference_streams(L, t, ub, 1000 * t + ub):
        used = C.c_uint64(enc.size)
        if L is not None:   # the real decoder first (sanity of the door itself)
            want = np.zeros(a.size, dtype=dt)
            assert L.ref_codec_decode(t, ub, enc.ctypes.data, enc.size, a.size, want.ctypes.data, C.byref(used)) == 0
            assert np.array_equal(want, a), (TYPES[t], ub, name, a.size)
        got = np.zeros(a.size, dtype=dt)
        cons = C.c_int64(0)
        padded = np.concatenate([enc, np.zeros(16, dtype=np.uint8)])     # decoders may not read past in_len
        r = O.ora_int_stream_decode(t, ub, padded.ctypes.data, enc.size, a.size, got.ctypes.data, C.byref(cons))
        assert r == 0, (TYPES[t], ub, name, a.size, r)
        assert np.array_equal(got, a), (TYPES[t], ub, name, a.size)
        assert cons.value == used.value == enc.size, (TYPES[t], ub, name, a.size, cons.value, used.value, enc.size)


@pytest.mark.parametrize("t", sorted(TYPES))
@pytest.mark.parametrize("ub", sorted(WIDTHS))
def test_writer_encoders_are_byte_exact(t, ub):
    """The writer's stream encoders (oceanbase_b200/csrc/stream_codecs_host.h) produce the reference encoders' bytes."""
    from oceanbase_b200.capi import lib
    for name, a, want in reference_streams(_ref(), t, ub, 77 * t + ub):
        v64 = np.ascontiguousarray(a.astype(np.uint64))
        n = C.c_int64(0)
        out = np.zeros(a.size * ub * 2 + 4096, dtype=np.uint8)
        r = lib.obgpu_writer_stream_encode(t, ub, v64.ctypes.data, a.size, out.ctypes.data, out.size, C.byref(n))
        assert r == 0
        assert n.value == want.size and np.array_equal(out[:n.value], want), (TYPES[t], ub, name, a.size, n.value, want.size)
