"""Phase B with codecs on the device (include/obgpu_compaction.h: obgpu_encode_columns_with, obgpu_merge_result_encode_with): with
DICT / RLE / CONST / INTEGER_BASE_DIFF forced, or OBGPU_ENC_AUTO choosing per micro-block, the device's blocks are byte for byte
the host writer's (sstable_writer.cpp: BlockBuilder::encode_* and choose_auto_encoding). A block the host writer refuses, or
writes with var-stored cells, reads size 0 and counts in n_host_blocks."""
import numpy as np
import pytest

import oracle_binding as ora
from test_encoder_selection import shapes as selection_shapes
from test_gpu_device_encoder import SHAPES, _ctx, _datum_len, device_encode, make_columns

pytestmark = pytest.mark.gpu

CODECS = {1: "DICT", 2: "RLE", 3: "CONST", 4: "INTEGER_BASE_DIFF"}
STORE_SIZE = {1: 1, 2: 2, 3: 4, 4: 4, 5: 8, 6: 1, 7: 2, 8: 4, 9: 4, 10: 8, 17: 8, 18: 8, 19: 4, 20: 8, 21: 1}   # type_store_size


def _cols(cols, encodings):
    from oceanbase_b200.sstable import Column
    return [Column(t, e, v, nulls=nl, byte_packing_only=bo) for (t, v, nl, bo), e in zip(cols, encodings)]


def encode_with(ctx, cols, encodings, rpb, rk, align=128):
    import torch
    from oceanbase_b200 import compaction
    keep, dcols = [], []
    for (t, v, nl, bo) in cols:
        dv = torch.from_numpy(v).cuda()
        dn = torch.from_numpy(nl).cuda() if nl is not None else None
        keep += [dv, dn]
        dcols.append((dv.data_ptr(), dn.data_ptr() if dn is not None else None, t, bo))
    return compaction.encode_columns(ctx, dcols, len(cols[0][1]), rpb, rowkey_cnt=rk, align=align, keep=keep, encodings=encodings)


def host_block_or_none(cols, encodings, row_begin, nrows, rk):
    """The host writer's block, or None where the device leaves it to the host writer: a refused codec, or var-stored cells."""
    from oceanbase_b200 import capi
    from oceanbase_b200.sstable import encode_block
    try:
        b = encode_block(_cols(cols, encodings), row_begin=row_begin, nrows=nrows, rowkey_cnt=rk)
    except capi.ObGpuError:
        return None
    return None if int(b[22]) | int(b[23]) else b   # opt2_: var-stored columns


def assert_blocks_match_host(enc, cols, encodings, rpb, rk, align=128):
    """Every block against the host writer's block of the same rows; offsets follow the aligned sizes. Returns the column
    codecs seen (from the column headers)."""
    img, off, sz = enc.fetch()
    n = len(cols[0][1])
    nb = (n + rpb - 1) // rpb
    assert len(off) == nb
    pos, host, seen = 0, 0, set()
    for b in range(nb):
        want = host_block_or_none(cols, encodings, b * rpb, min(rpb, n - b * rpb), rk)
        assert off[b] == pos, (b, off[b], pos)
        if want is None:
            assert sz[b] == 0, b
            host += 1
            continue
        got = img[off[b]:off[b] + sz[b]]
        if not np.array_equal(got, want):
            bad = int(np.nonzero(got[:min(len(got), len(want))] != want[:min(len(got), len(want))])[0][0]) if len(got) and len(want) else -1
            raise AssertionError(f"block {b}: device {len(got)} bytes, host {len(want)} bytes, first differing byte {bad}")
        seen |= {int(want[64 + 16 * c + 1]) for c in range(len(cols))}
        pos += (int(sz[b]) + align - 1) // align * align
    assert enc.info().n_host_blocks == host
    assert enc.info().image_size == pos
    return seen


def assert_oracle_accepts(enc, cols, rpb, blocks=None):
    img, off, sz = enc.fetch()
    blocks = range(len(off)) if blocks is None else blocks
    for b in blocks:
        if sz[b] == 0:
            continue
        blk = ora.Block(img[off[b]:off[b] + sz[b]].copy())
        assert blk.verify_checksums() == 0
        for c, (t, v, nl, _bo) in enumerate(cols):
            for r in range(0, int(blk.row_count), max(1, int(blk.row_count) // 13)):
                cell = blk.cell(c, r)
                if nl is not None and nl[b * rpb + r]:
                    assert cell is None, (b, c, r)
                else:
                    mask = (1 << (8 * STORE_SIZE[t])) - 1
                    assert (int(cell) & mask) == (int(v[b * rpb + r]) & mask), (b, c, r)
    o = ora.oracle()
    got = enc.column_checksums()
    n = len(cols[0][1])
    for c, (t, v, nl, _bo) in enumerate(cols):
        assert int(got[c]) == o.ora_column_checksum(v.ctypes.data, nl.ctypes.data if nl is not None else None, n, _datum_len(t)), c


def _low_card_and_runs(rng):
    """Low-cardinality and run-heavy variants of the SHAPES columns."""
    from oceanbase_b200 import capi
    out = []
    n = 6_000
    pool = rng.integers(-(1 << 40), 1 << 40, size=5)
    low = pool[rng.integers(0, 5, size=n)].astype(np.int64)
    runs = np.repeat(rng.integers(0, 1 << 20, size=n // 40 + 1), 40)[:n].astype(np.int64)
    nearly = np.full(n, 123_456, dtype=np.int64)
    nearly[rng.choice(n, size=n // 200, replace=False)] = rng.integers(0, 1000, size=n // 200)
    nl = (rng.random(n) < 0.1).astype(np.uint8)
    cols = [(capi.OBJ_INT, low, None, False), (capi.OBJ_INT, runs, nl, False), (capi.OBJ_INT, nearly, None, False),
            (capi.OBJ_UINT32, (runs & 0xffffffff).astype(np.int64), None, True), (capi.OBJ_DATE, (low & 0xfff) + 8000, None, False),
            (capi.OBJ_TINYINT, ((low & 0xff) - 128).astype(np.int64), nl, False)]
    out.append(("low_card_runs", cols, n, 500, 1))
    # constant columns (one value per block, all-NULL blocks)
    c = np.repeat(rng.integers(0, 1 << 30, size=n // 300 + 1), 300)[:n].astype(np.int64)
    an = np.zeros(n, dtype=np.uint8)
    an[900:1200] = 1
    out.append(("constants", [(capi.OBJ_INT, c, None, False), (capi.OBJ_INT, c, an, False), (capi.OBJ_YEAR, (c & 0x7f), None, False)], n, 300, 0))
    return out


def _forced_cases():
    rng = np.random.default_rng(21)
    cases = []
    for i, (name, spec, n, rpb, rk) in enumerate(SHAPES):
        cases.append((name, make_columns(np.random.default_rng(31 + i), n, spec), n, rpb, rk))
    return cases + _low_card_and_runs(rng)


@pytest.mark.parametrize("codec", sorted(CODECS), ids=[CODECS[c] for c in sorted(CODECS)])
def test_forced_codecs_equal_the_host_writer(codec):
    ctx = _ctx()
    for name, cols, n, rpb, rk in _forced_cases():
        encodings = [codec] * len(cols)
        enc = encode_with(ctx, cols, encodings, rpb, rk)
        assert_blocks_match_host(enc, cols, encodings, rpb, rk)
        assert_oracle_accepts(enc, cols, rpb, blocks=(0, len(enc.fetch()[1]) // 2, len(enc.fetch()[1]) - 1))
        enc.free()


@pytest.mark.parametrize("align", [16, 128, 4096])
def test_alignments_and_block_sizes(align):
    from oceanbase_b200 import capi
    ctx = _ctx()
    rng = np.random.default_rng(align)
    cols = make_columns(rng, 9_000, [(5, 45, 0.0, False), (5, 64, 0.1, False), (5, 10, 0.0, False), (5, 27, 0.02, False)])
    cols[2] = (cols[2][0], cols[2][1] % 7, None, False)
    for rpb in (1, 700, 4096):
        m = 200 if rpb == 1 else len(cols[0][1])
        k = 2 if rpb == 4096 else 4   # four AUTO columns of 4096 rows do not fit one CTA's shared memory
        sub = [(t, v[:m].copy(), None if nl is None else nl[:m].copy(), bo) for (t, v, nl, bo) in cols[:k]]
        for encodings in ([capi.ENC_AUTO] * k, [capi.ENC_INTEGER_BASE_DIFF, capi.ENC_RAW, capi.ENC_DICT, capi.ENC_RLE][:k]):
            enc = encode_with(ctx, sub, encodings, rpb, 1, align=align)
            assert_blocks_match_host(enc, sub, encodings, rpb, 1, align=align)
            enc.free()


def _auto_table(cols, rpb, rk, align=128):
    from oceanbase_b200 import capi
    from oceanbase_b200.sstable import encode_table
    return encode_table(_cols(cols, [capi.ENC_AUTO] * len(cols)), rpb, rowkey_cnt=rk, align=align)


def _assert_auto_image(enc, table, n_cols):
    img, off, sz = enc.fetch()
    assert enc.info().n_host_blocks == 0
    assert np.array_equal(off, np.asarray(table.offsets)) and np.array_equal(sz, np.asarray(table.sizes))
    want = np.asarray(table.image)
    if not np.array_equal(img, want):
        bad = int(np.nonzero(img != want)[0][0]) if img.size == want.size else -1
        raise AssertionError(f"AUTO image differs from the host writer's (first differing byte {bad})")
    return {int(want[o + 64 + 16 * c + 1]) for o in off for c in range(n_cols)}


def test_auto_equals_the_host_writer():
    from oceanbase_b200 import capi
    ctx = _ctx()
    seen = set()
    # the shapes of the host writer's selection test, one column each
    for n in (1000, 257):
        for name, (v, nl, _want) in selection_shapes(n, np.random.default_rng(11)).items():
            cols = [(capi.OBJ_INT, v, nl, False)]
            for rpb in (n, 97):
                enc = encode_with(ctx, cols, [capi.ENC_AUTO], rpb, 0)
                seen |= _assert_auto_image(enc, _auto_table(cols, rpb, 0), 1)
                assert_oracle_accepts(enc, cols, rpb)
                enc.free()
    # random columns drawn as the host writer's round-trip test draws them (NULL cells only: merged rows have no NOP)
    rng = np.random.default_rng(13)
    for trial in range(120):
        n = int(rng.integers(1, 600))
        card = int(rng.choice([1, 2, 5, 50, 10_000]))
        bits = int(rng.choice([1, 7, 16, 33, 62]))
        pool = rng.integers(0, 1 << bits, size=card, dtype=np.int64) + int(rng.choice([0, 10**9, -(1 << 40)]))
        v = pool[rng.integers(0, card, size=n)]
        if rng.random() < 0.4:
            v = np.sort(v)
        nl = (rng.random(n) < rng.choice([0.0, 0.1, 0.9])).astype(np.uint8)
        nl = nl if nl.any() else None
        t = int(rng.choice([capi.OBJ_INT, capi.OBJ_UINT64])) if v.min() >= 0 else capi.OBJ_INT
        cols = [(t, v, nl, False)]
        enc = encode_with(ctx, cols, [capi.ENC_AUTO], n, 0)
        table = _auto_table(cols, n, 0)
        if int(table.block(0)[22]) | int(table.block(0)[23]):   # the host chose var-stored RAW: left to it
            assert enc.fetch()[2][0] == 0 and enc.info().n_host_blocks == 1, trial
        else:
            seen |= _assert_auto_image(enc, table, 1)
        enc.free()
    # a mixed multi-column table
    mixed = make_columns(np.random.default_rng(3), 20_000, [(5, 40, 0.0, False), (4, 32, 0.2, False), (19, 20, 0.1, False),
                                                             (21, 8, 0.0, False), (10, 64, 0.0, True), (1, 8, 0.1, False)])
    mixed[0] = (5, np.arange(20_000, dtype=np.int64) * 5 + 10**9, None, False)
    mixed[3] = (21, mixed[3][1] % 3, None, False)
    enc = encode_with(ctx, mixed, [capi.ENC_AUTO] * len(mixed), 700, 1)
    seen |= _assert_auto_image(enc, _auto_table(mixed, 700, 1), len(mixed))
    assert_oracle_accepts(enc, mixed, 700, blocks=(0, 13, 28))
    enc.free()
    assert seen >= {0, 1, 2, 3, 4}, seen


@pytest.mark.parametrize("shape", ["cfg5", "lineitem", "eventlog"])
def test_auto_on_the_benchmark_shapes(shape):
    from oceanbase_b200 import capi, compaction
    from oceanbase_b200.synth import make_encode_columns
    ctx = _ctx()
    n, rpb = 200_000, 500
    dcols = make_encode_columns(shape, n, seed=5)
    cols = [(t, v.cpu().numpy(), None if nl is None else nl.cpu().numpy(), False) for (t, v, nl) in dcols]
    enc = compaction.encode_columns(ctx, [(v.data_ptr(), None if nl is None else nl.data_ptr(), t, False) for (t, v, nl) in dcols], n, rpb,
                                    rowkey_cnt=1, keep=dcols, encodings=[capi.ENC_AUTO] * len(cols))
    seen = _assert_auto_image(enc, _auto_table(cols, rpb, 1), len(cols))
    assert_oracle_accepts(enc, cols, rpb, blocks=(0, 200, 399))
    if shape == "eventlog":
        assert seen == {0, 1, 3, 4}, seen
    raw = compaction.encode_columns(ctx, [(v.data_ptr(), None if nl is None else nl.data_ptr(), t, False) for (t, v, nl) in dcols], n, rpb,
                                    rowkey_cnt=1, keep=dcols)
    assert enc.info().image_size < raw.info().image_size
    enc.free()
    raw.free()


def test_null_dominated_block_under_auto():
    """The block test_null_dominated_column_is_left_to_the_host leaves to the host writer under RAW: under AUTO the device
    encodes it whenever the host writer's AUTO does not pick (var-stored) RAW for it."""
    from oceanbase_b200 import capi
    ctx = _ctx()
    rng = np.random.default_rng(6)
    n, rpb = 4_000, 500
    cols = make_columns(rng, n, [(5, 30, 0.0, False), (5, 60, 0.0, False)])
    nl = np.zeros(n, dtype=np.uint8)
    nl[1000:1500] = 1
    nl[1500:2000:2] = 1
    cols[1] = (cols[1][0], cols[1][1], nl, False)
    raw, _ = device_encode(ctx, cols, rpb, 1)
    assert raw.info().n_host_blocks == 1
    enc = encode_with(ctx, cols, [capi.ENC_AUTO] * 2, rpb, 1)
    assert_blocks_match_host(enc, cols, [capi.ENC_AUTO] * 2, rpb, 1)
    table = _auto_table(cols, rpb, 1)
    host_var = sum(1 for b in range(table.n_blocks) if int(table.block(b)[22]) | int(table.block(b)[23]))
    assert enc.info().n_host_blocks == host_var
    assert enc.info().n_host_blocks < raw.info().n_host_blocks
    enc.free()
    raw.free()


def test_merge_result_with_auto_encodings():
    """co_merge_write with every column AUTO on the three-run merge of test_column_groups_of_a_merge_result: each group equals the
    host writer's AUTO image of the oracle's merged rows, and the device image re-opens as a page batch that scans like the host
    image."""
    import torch
    import oceanbase_b200 as ob
    from oceanbase_b200 import capi, compaction
    from oceanbase_b200.sstable import Column, TableImage, encode_table
    ctx = _ctx()
    rng = np.random.default_rng(9)
    runs, oruns = [], []
    for r in range(3):
        n = 6_000
        key = np.sort(rng.choice(40_000, size=n, replace=False)).astype(np.int64)
        cols = [Column(capi.OBJ_INT, capi.ENC_INTEGER_BASE_DIFF, key)]
        vals, ext = [], []
        for c in range(3):
            v = rng.integers(0, 1 << (10 + 17 * c), size=n, dtype=np.int64)
            nl = (rng.random(n) < 0.1).astype(np.uint8) if c == 1 else None
            cols.append(Column(capi.OBJ_INT, capi.ENC_RAW, v, nulls=nl))
            vals.append(v)
            ext.append(nl if nl is not None else np.zeros(n, dtype=np.uint8))
        runs.append(encode_table(cols, 700, rowkey_cnt=1))
        oruns.append({"key": key, "flag": None, "vals": vals, "ext": ext})
    want = ora.major_merge(oruns, 3)
    batches = [ob.PageBatch(ctx, t) for t in runs]
    res = compaction.merge_batches(ctx, batches, 0, None, [1, 2, 3])
    groups = [[-1, 0, 1, 2], [0], [1], [2, 0]]
    types = {-1: capi.OBJ_INT, 0: capi.OBJ_INT, 1: capi.OBJ_INT, 2: capi.OBJ_INT}
    encs = compaction.co_merge_write(res, groups, types, rows_per_block=900, encodings={c: capi.ENC_AUTO for c in types})
    for cg, enc in zip(groups, encs):
        host_cols = []
        for c in cg:
            if c == -1:
                host_cols.append(Column(capi.OBJ_INT, capi.ENC_AUTO, want["key"]))
            else:
                nl = want["null"][c]
                host_cols.append(Column(capi.OBJ_INT, capi.ENC_AUTO, want["vals"][c], nulls=nl if nl.any() else None))
        table = encode_table(host_cols, 900, rowkey_cnt=1 if cg[0] == -1 else 0)
        _assert_auto_image(enc, table, len(cg))
        if cg[0] == -1:
            d_img, d_off, _ = enc.device_image()
            img, off, sz = enc.fetch()
            dev_table = TableImage(img, off, sz, table.total_rows, len(cg))
            flt = ob.White(1, ob.WHITE_OP_LT, (1 << 9,))
            a = ctx.open_batch(dev_table, device_image_ptr=d_img, host_view=False, image_size=img.size)
            b = ctx.open_batch(table)
            ra, rb = a.scan(flt, list(range(len(cg))), want_row_ids=True), b.scan(flt, list(range(len(cg))), want_row_ids=True)
            assert ra.selected_rows == rb.selected_rows and ra.selected_rows > 0
            assert np.array_equal(ra.fetch_row_ids(), rb.fetch_row_ids())
            for i in range(len(cg)):
                da, _, na = ra.fetch_col(i)
                db, _, nb = rb.fetch_col(i)
                assert np.array_equal(da, db) and np.array_equal(na, nb), i
            ra.free(); rb.free(); a.close(); b.close()
        enc.free()
    torch.cuda.synchronize()


def test_call_level_refusals():
    import torch
    from oceanbase_b200 import capi, compaction
    ctx = _ctx()
    n = 10_000
    v = torch.arange(n, device="cuda", dtype=torch.int64)
    col = (v.data_ptr(), None, capi.OBJ_INT, False)
    with pytest.raises(capi.ObGpuError) as ei:   # a string column
        compaction.encode_columns(ctx, [col, (v.data_ptr(), None, capi.OBJ_VARCHAR, False)], n, 500, encodings=[capi.ENC_AUTO, capi.ENC_RAW])
    assert ei.value.code == capi.OB_NOT_SUPPORTED
    import ctypes as C
    bad = np.array([7], dtype=np.int32)   # an encoding outside the six, past the Python wrapper's own check
    h = C.c_void_p()
    assert capi.lib.obgpu_encode_columns_with(ctx._h, compaction._encode_cols([col]), bad.ctypes.data, 1, 0, n, 500, 128,
                                              C.byref(h)) == capi.OB_INVALID_ARGUMENT
    with pytest.raises(capi.ObGpuError) as ei:   # rows_per_block above the codec kernel's cap
        compaction.encode_columns(ctx, [col], n, 4097, encodings=[capi.ENC_DICT])
    assert ei.value.code == capi.OB_NOT_SUPPORTED
    raw = compaction.encode_columns(ctx, [col], n, 4097, encodings=[capi.ENC_RAW])   # RAW keeps the RAW encoder's limits
    assert raw.info().n_blocks == 3
    raw.free()
    with pytest.raises(capi.ObGpuError) as ei:   # the requested codecs' largest block does not fit shared memory
        compaction.encode_columns(ctx, [col] * 4, n, 4096, encodings=[capi.ENC_AUTO] * 4)
    assert ei.value.code == capi.OB_NOT_SUPPORTED
    ok = compaction.encode_columns(ctx, [col] * 4, n, 4096)   # ... while RAW still takes it
    ok.free()
