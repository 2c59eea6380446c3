"""Seeded synthetic SSTables of the BASELINE.json configs (SURVEY.md 8d).

Every column is generated from SplitMix64(seed, column) so any slice of a table can be regenerated
independently (ranks generate their own shard without communication). Compressor none, PAX
ENCODING_ROW_STORE blocks produced by the host writer.
"""
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import capi
from .scan import White, And
from .sstable import Column, TableImage, encode_table

_M64 = (1 << 64) - 1


def splitmix64(seed: int, start: int, n: int) -> np.ndarray:
    """n SplitMix64 outputs for counters start .. start+n-1 (stateless form: hash of seed+ctr*gamma)."""
    with np.errstate(over="ignore"):
        idx = np.arange(start + 1, start + n + 1, dtype=np.uint64)
        z = np.uint64(seed & _M64) + idx * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _col_seed(seed, col):
    return (seed * 0x100000001B3 + col * 0x9E3779B1 + 12345) & _M64


@dataclass
class Workload:
    table: TableImage
    filter: object
    proj: List[int]
    proj_is_string: List[bool]
    proj_elem_len: List[int]
    name: str
    rows_per_block: int
    # algorithmic bytes per input row (SURVEY.md 8d): B_in = encoded bytes, B_out = dense output
    def alg_bytes(self, selected_rows: int) -> int:
        out_per_row = sum(12 if s else l for s, l in zip(self.proj_is_string, self.proj_elem_len))
        bitmap = (self.table.total_rows + 7) // 8
        return int(self.table.sizes.sum()) + selected_rows * out_per_row + bitmap


# ---- config 1: 4 x INT64, RAW fixed 8 B, no filter -------------------------------------------------
def make_config1(rows=1_000_000, rows_per_block=500, seed=1, row_start=0) -> Workload:
    cols = []
    for c in range(4):
        v = splitmix64(_col_seed(seed, c), row_start, rows).view(np.int64)
        cols.append(Column(capi.OBJ_INT, capi.ENC_RAW, v))
    table = encode_table(cols, rows_per_block)
    return Workload(table, None, [0, 1, 2, 3], [False] * 4, [8] * 4, "cfg1: 4xINT64 RAW, no filter", rows_per_block)


# ---- config 2: 8 x INT64, base-diff PK + 3 RLE + 4 bit-packed RAW, one range predicate ---------------
def _rle_column(seed, start, n, dict_bits=8, mean_run=64):
    """Runs with geometric length (mean `mean_run`) over a 2^dict_bits value dictionary. Run
    boundaries are a pure function of the row index so shards line up."""
    h = splitmix64(seed, start, n)
    # a row starts a new run with probability 1/mean_run
    boundary = (h % np.uint64(mean_run)) == 0
    if n:
        boundary[0] = True
    run_id = np.cumsum(boundary) - 1
    starts = np.flatnonzero(boundary)
    # value of a run: hash of the absolute row index of its first row
    run_vals = splitmix64(seed ^ 0xABCDEF, 0, 1)[0] ^ splitmix64(seed + 17, 0, 1)[0]
    hv = splitmix64(seed + 99, start, n)[starts]
    vals = (hv ^ run_vals) & np.uint64((1 << dict_bits) - 1)
    # spread dictionary values over a wide integer range so the dict stores multi-byte values
    wide = (vals.astype(np.int64) * 1_000_003 + 7)
    return wide[run_id]


def config2_pk(rows, seed, row_start=0):
    """Sorted PK of the config-2 table as a pure function of the absolute row index (shards / chunks line up,
    strictly increasing: consecutive rows differ by 351 + (j' - j) with j, j' in [0, 351))."""
    jitter = (splitmix64(_col_seed(seed, 0), row_start, rows) % np.uint64(351)).astype(np.int64)
    return np.int64(1_000_000_007) + (np.arange(row_start, row_start + rows, dtype=np.int64)) * 351 + jitter


def config2_columns(rows, seed, row_start=0):
    """The 8 INT64 columns of a config-2 chunk (the values the encoded table must decode back to)."""
    s = lambda c: _col_seed(seed, c)
    vals = [config2_pk(rows, seed, row_start)]
    for c in (1, 2, 3):
        vals.append(_rle_column(s(c), row_start, rows))
    for c, w in zip((4, 5, 6, 7), (7, 13, 21, 33)):
        vals.append((splitmix64(s(c), row_start, rows) & np.uint64((1 << w) - 1)).astype(np.int64))
    return vals


def make_config2_like(rows=100_000, rows_per_block=1400, seed=2, shape="bt", row_start=0,
                      n_threads=0, out=None) -> Workload:
    vals = config2_columns(rows, seed, row_start)
    encs = [capi.ENC_INTEGER_BASE_DIFF] + [capi.ENC_RLE] * 3 + [capi.ENC_RAW] * 4
    cols = [Column(capi.OBJ_INT, e, v) for e, v in zip(encs, vals)]
    table = encode_table(cols, rows_per_block, rowkey_cnt=1, n_threads=n_threads, out=out)
    if shape == "bt":
        flt = White(4, capi.WHITE_OP_BT, (32, 63))                      # 32/128 = 25 %
    else:
        flt = And([White(4, capi.WHITE_OP_GE, (32,)), White(4, capi.WHITE_OP_LE, (63,))])
    return Workload(table, flt, list(range(8)), [False] * 8, [8] * 8,
                    f"cfg2: 8xINT64 base-diff PK + 3 RLE + 4 bit-packed RAW, range predicate ({shape}) 25%",
                    rows_per_block)


# ---- config 3: 8 INT64 DICT + 8 VARCHAR DICT, 3-predicate AND ~10 % --------------------------------
def _zipf_ranks(seed, start, n, card, a=1.1):
    """Zipf(a) ranks in [0, card) by inverse CDF over a precomputed table."""
    w = 1.0 / np.power(np.arange(1, card + 1, dtype=np.float64), a)
    cdf = np.cumsum(w)
    cdf /= cdf[-1]
    u = (splitmix64(seed, start, n) >> np.uint64(11)).astype(np.float64) / float(1 << 53)
    return np.searchsorted(cdf, u, side="left").astype(np.int64)


def _string_dict(seed, card, min_len=8, max_len=32):
    h = splitmix64(seed, 0, card)
    lens = (h % np.uint64(max_len - min_len + 1)).astype(np.int64) + min_len
    off = np.zeros(card + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    raw = splitmix64(seed + 1, 0, int(off[-1]))
    heap = (raw % np.uint64(26)).astype(np.uint8) + ord("a")
    return heap, off


def make_config3_like(rows=100_000, rows_per_block=1100, seed=3, row_start=0, n_threads=0, out=None) -> Workload:
    s = lambda c: _col_seed(seed, c)
    int_cards = [16, 64, 256, 4096, 16, 1024, 65536, 200]
    cols = []
    for c, card in enumerate(int_cards):
        r = _zipf_ranks(s(c), row_start, rows, card)
        # dictionary value of rank k: wide multi-byte integers, shard independent
        vals = (splitmix64(s(c) + 5, 0, card) >> np.uint64(20)).astype(np.int64)
        if c == 3:
            vals = np.arange(card, dtype=np.int64) * 1000  # ordered domain for the `<` predicate
        cols.append(Column(capi.OBJ_INT, capi.ENC_DICT, vals[r]))
    str_dicts = []
    for c in range(8, 16):
        card = 1024
        heap, off = _string_dict(s(c) + 3, card)
        r = _zipf_ranks(s(c), row_start, rows, card)
        lens = off[1:] - off[:-1]
        rl = lens[r]
        roff = np.zeros(rows + 1, dtype=np.int64)
        np.cumsum(rl, out=roff[1:])
        # gather bytes: index arithmetic without a python loop
        idx = np.repeat(off[:-1][r] - roff[:-1], rl) + np.arange(roff[-1], dtype=np.int64)
        cols.append(Column(capi.OBJ_VARCHAR, capi.ENC_DICT, None, str_heap=heap[idx], str_off=roff))
        str_dicts.append((heap, off))
    table = encode_table(cols, rows_per_block, n_threads=n_threads, out=out)
    # c0 = k  (Zipf rank 0 of 16: ~30 %), c3 < v, s1 IN (5 strings): tuned to ~10 % combined
    c0_vals = (splitmix64(s(0) + 5, 0, 16) >> np.uint64(20)).astype(np.int64)
    heap9, off9 = str_dicts[1]
    in_list = tuple(bytes(heap9[off9[k]:off9[k + 1]]) for k in (0, 1, 2, 3, 5))
    flt = And([White(0, capi.WHITE_OP_EQ, (int(c0_vals[0]),)),
               White(3, capi.WHITE_OP_LT, (2_000_000,)),
               White(9, capi.WHITE_OP_IN, in_list)])
    proj = [1, 2, 5, 6, 8, 10]
    return Workload(table, flt, proj, [False] * 4 + [True] * 2, [8] * 4 + [8] * 2,
                    "cfg3: 8 INT64 DICT + 8 VARCHAR DICT, 3-predicate AND", rows_per_block)


# ---- config 5: K sorted runs with overlapping rowkey ranges (major compaction input) -----------------
def make_config5_runs(n_runs=8, window=100_000, seed=5, rows_per_block=1400, dup_pct=10, delete_pct=2,
                      nop_pct=50, null_pct=5, n_threads=0, encode=True, only=None):
    """Run r (0 = oldest table) covers rowkey indexes [r * window / 2, r * window / 2 + window): adjacent runs
    overlap by 50 %. A rowkey index lives in one covering run (its home, chosen by hash); dup_pct % of the
    indexes are present in EVERY covering run (newer copies are DF_UPDATE rows whose payload cells are NOP
    with probability nop_pct %), delete_pct % of the rows of runs >= 1 are DF_DELETE rows (payload NOP).
    Columns of a run's SSTable: 0 rowkey INT64 (INTEGER_BASE_DIFF), 1 ObDmlFlag (TINYINT RAW), 2..4 payload
    INT64 (RAW, NULL / NOP as ext values). Returns a list of dicts: key, flag, vals[3], ext[3] (numpy) and
    `table` (TableImage) when encode."""
    runs = []
    for r in range(n_runs):
        if only is not None and r not in only:   # a rank of a multi-GPU job generates the runs it holds (a run is a pure function of r)
            runs.append(None)
            continue
        lo = r * (window // 2)
        i = np.arange(lo, lo + window, dtype=np.int64)
        h = splitmix64(_col_seed(seed, 100), int(lo), window)           # pure function of the rowkey index
        # covering runs of index i: those r' with r' * window/2 <= i < r' * window/2 + window
        first_cov = np.maximum((i - window) // (window // 2) + 1, 0)
        last_cov = np.minimum(i // (window // 2), n_runs - 1)
        ncov = (last_cov - first_cov + 1).astype(np.uint64)
        home = first_cov + (h % ncov).astype(np.int64)
        dup = ((h >> np.uint64(20)) % np.uint64(100)) < np.uint64(dup_pct)
        present = (home == r) | dup
        idx = i[present]
        hh = h[present]
        key = np.int64(1_000_003) + idx * 5 + (hh % np.uint64(5)).astype(np.int64)
        n = len(key)
        newer_copy = dup[present] & (first_cov[present] < r)            # an older covering run holds this key too
        hr = splitmix64(_col_seed(seed, 200 + r), int(lo), window)[present]
        flag = np.full(n, capi.DF_INSERT, dtype=np.uint8)
        flag[newer_copy] = capi.DF_UPDATE
        is_del = (r >= 1) & (((hr >> np.uint64(8)) % np.uint64(100)) < np.uint64(delete_pct))
        flag[is_del] = capi.DF_DELETE
        vals, ext = [], []
        for c in range(3):
            hv = splitmix64(_col_seed(seed, 300 + 10 * r + c), int(lo), window)[present]
            v = (hv >> np.uint64(24)).astype(np.int64)
            e = np.zeros(n, dtype=np.uint8)
            e[((hv % np.uint64(100)) < np.uint64(null_pct))] = 1
            e[newer_copy & (((hv >> np.uint64(7)) % np.uint64(100)) < np.uint64(nop_pct))] = 2
            e[flag == capi.DF_DELETE] = 2
            v[e != 0] = 0
            vals.append(v)
            ext.append(e)
        run = {"key": key, "flag": flag, "vals": vals, "ext": ext}
        if encode:
            cols = [Column(capi.OBJ_INT, capi.ENC_INTEGER_BASE_DIFF, key),
                    Column(capi.OBJ_TINYINT, capi.ENC_RAW, flag.astype(np.int64))]
            for c in range(3):
                cols.append(Column(capi.OBJ_INT, capi.ENC_RAW, vals[c], nulls=ext[c] if ext[c].any() else None))
            run["table"] = encode_table(cols, rows_per_block, rowkey_cnt=1, n_threads=n_threads)
        runs.append(run)
    return runs


# ---- config 4: TPC-H lineitem columns of Q6 as a CS_ENCODING_ROW_STORE column group -----------------
Q6_DATE_LO, Q6_DATE_HI = 8766, 9131        # 1994-01-01 <= l_shipdate < 1995-01-01 (days since 1970-01-01)


def make_config4_like(rows=100_000, rows_per_block=2000, seed=4, row_start=0, n_threads=0) -> Workload:
    """dbgen-shaped value domains (TPC-H spec 4.2.3): l_shipdate uniform in [1992-01-02, 1998-12-01], l_discount
    0.00..0.10 (stored x100), l_quantity 1..50, l_extendedprice = quantity x part retail price (90 000..200 000
    cents, stored as decimal-int cents). Columns: 0 l_shipdate (DATE), 1 l_discount, 2 l_quantity,
    3 l_extendedprice, all CS INTEGER. Filter = Q6, projection = (l_extendedprice, l_discount)."""
    s = lambda c: _col_seed(seed, c)
    shipdate = (splitmix64(s(0), row_start, rows) % np.uint64(2526)).astype(np.int64) + 8036
    discount = (splitmix64(s(1), row_start, rows) % np.uint64(11)).astype(np.int64)
    quantity = (splitmix64(s(2), row_start, rows) % np.uint64(50)).astype(np.int64) + 1
    retail = (splitmix64(s(3), row_start, rows) % np.uint64(110_001)).astype(np.int64) + 90_000
    price = quantity * retail
    cols = [Column(capi.OBJ_DATE, capi.ENC_CS_INTEGER, shipdate), Column(capi.OBJ_INT, capi.ENC_CS_INTEGER, discount),
            Column(capi.OBJ_INT, capi.ENC_CS_INTEGER, quantity), Column(capi.OBJ_INT, capi.ENC_CS_INTEGER, price)]
    table = encode_table(cols, rows_per_block, n_threads=n_threads)
    flt = And([White(0, capi.WHITE_OP_GE, (Q6_DATE_LO,)), White(0, capi.WHITE_OP_LT, (Q6_DATE_HI,)),
               White(1, capi.WHITE_OP_BT, (5, 7)), White(2, capi.WHITE_OP_LT, (24,))])
    return Workload(table, flt, [3, 1], [False, False], [8, 8],
                    "cfg4: TPC-H lineitem Q6 columns as a CS column group (4 CS INTEGER columns), Q6 predicate, SUM(price*discount)",
                    rows_per_block)


# ---- micro-block size target ------------------------------------------------------------------------------
MICRO_BLOCK_TARGET = 16 << 10   # OB_DEFAULT_SSTABLE_BLOCK_SIZE (deps/oblib/src/lib/ob_define.h:1988)


def rows_per_block_for_target(maker, target_bytes=MICRO_BLOCK_TARGET, sample_rows=40_000, seed=None, lo=16, hi=8192):
    """Rows per micro-block at which `maker`'s table cuts blocks of (on average) at most `target_bytes` encoded
    bytes. The reference's encoder cuts a block when the running size estimate reaches the limit and corrects the
    estimate with the previous block's real / estimated ratio (ObMicroBlockEncoder::update_estimate_size_limit,
    encoding/ob_micro_block_encoder.cpp:357-381), i.e. it converges on blocks of about the target size; the
    synthetic tables have stationary columns, so a constant row count per block is that steady state. Found by
    bisection on a seeded sample."""
    kw = {} if seed is None else {"seed": seed}

    def mean_block(rpb):
        w = maker(rows=max(sample_rows, rpb * 8), rows_per_block=rpb, **kw)
        n_full = max(1, w.table.n_blocks - 1)   # the ragged last block does not count
        return float(w.table.sizes[:n_full].mean())

    if mean_block(lo) > target_bytes:
        return lo
    while lo + 1 < hi:
        mid = (lo + hi) // 2
        if mean_block(mid) <= target_bytes:
            lo = mid
        else:
            hi = mid
    return lo


def referenced_bytes(table: TableImage, cols) -> int:
    """Bytes of the blocks' accessed regions for a scan that references `cols` (SURVEY.md 8d, B_in): per PAX block
    the 64-byte header + the column headers + the region [offset_c, offset_{c+1}) of the column area for every
    referenced column (meta + values / refs + dictionary: exactly what the kernels stage). Blocks with var-stored
    columns (row data) or CS blocks count whole."""
    img, total = table.image, 0
    cols = sorted(set(int(c) for c in cols))
    offs = np.asarray(table.offsets, dtype=np.int64)
    sizes = np.asarray(table.sizes, dtype=np.int64)
    hdr = np.stack([img[offs + k] for k in range(28)], axis=1).astype(np.int64)
    u16 = lambda a: hdr[:, a] | (hdr[:, a + 1] << 8)
    u32 = lambda a: hdr[:, a] | (hdr[:, a + 1] << 8) | (hdr[:, a + 2] << 16) | (hdr[:, a + 3] << 24)
    header_size, ncol, rst, var_cols, row_data_off = u32(4), u16(10), hdr[:, 20], u16(22), u32(24)
    whole = (rst == 3) | (var_cols > 0)     # CS_ENCODING_ROW_STORE / var-stored columns: no per-column region
    total += int(sizes[whole].sum())
    sel = ~whole
    if sel.any():
        o, hs, nc, rdo = offs[sel], header_size[sel], ncol[sel], row_data_off[sel]
        meta = hs + 16 * nc

        def col_off(c):
            b = o + hs + 16 * c + 8
            return (img[b].astype(np.int64) | (img[b + 1].astype(np.int64) << 8) | (img[b + 2].astype(np.int64) << 16) |
                    (img[b + 3].astype(np.int64) << 24))
        total += int(meta.sum())
        for c in cols:
            start = col_off(c)
            nxt = np.where(c + 1 < nc, col_off(np.minimum(c + 1, nc - 1)), rdo - meta)
            total += int((nxt - start).sum())
    return total


def filter_columns(expr):
    """Store indexes of the columns a filter tree references."""
    if expr is None:
        return []
    if isinstance(expr, White):
        return [expr.col]
    out = []
    for c in expr.children:
        out += filter_columns(c)
    return sorted(set(out))


# ---- device encoder shapes (tools/bench_encode.py, tests/test_gpu_device_encoder_codecs.py) ------------------------------------
ENCODE_SHAPES = ("cfg5", "lineitem", "eventlog")


def make_encode_columns(shape: str, n: int, seed: int = 5, device="cuda"):
    """Integer columns for the device encoder, generated with torch on `device` from `seed`, rowkey first:
    [(OBJ_* type, int64 values, uint8 NULL bytes or None)].
      cfg5     : key = 3 i + 1e9 + 7; 33-bit; 63-bit signed; 13-bit with 5 % NULLs
      lineitem : sorted orderkey with up to 4 lines an order; quantity 1..50; discount 0..10; tax 0..8; DATE over 2 526 days;
                 price; a 3-value status in runs of 50 rows
      eventlog : DATETIME in microseconds, increasing; 8 tenant ids of up to 900 123; HTTP status 97 % 200; user id in a 10^6
                 range above 10^12; 20-bit latency"""
    import torch
    g = torch.Generator(device=device).manual_seed(seed)

    def rnd(lo, hi):
        return torch.randint(lo, hi, (n,), device=device, dtype=torch.int64, generator=g)

    i = torch.arange(n, device=device, dtype=torch.int64)
    if shape == "cfg5":
        nl = (torch.rand((n,), device=device, generator=g) < 0.05).to(torch.uint8)
        return [(capi.OBJ_INT, i * 3 + 1_000_000_007, None), (capi.OBJ_INT, rnd(0, 1 << 33), None),
                (capi.OBJ_INT, rnd(-(1 << 62), 1 << 62), None), (capi.OBJ_INT, rnd(0, 1 << 13), nl)]
    if shape == "lineitem":
        orderkey = torch.cumsum((torch.rand((n,), device=device, generator=g) < 0.25).to(torch.int64), 0) * 32 + 1   # ~4 lines an order
        runs = torch.randint(0, 3, ((n + 49) // 50,), device=device, dtype=torch.int64, generator=g)
        status = torch.tensor([70, 79, 80], device=device, dtype=torch.int64)[runs].repeat_interleave(50)[:n]
        return [(capi.OBJ_INT, orderkey, None), (capi.OBJ_INT, rnd(1, 51), None), (capi.OBJ_INT, rnd(0, 11), None),
                (capi.OBJ_INT, rnd(0, 9), None), (capi.OBJ_DATE, rnd(8035, 8035 + 2526), None), (capi.OBJ_INT, rnd(90_000, 10_500_000), None),
                (capi.OBJ_INT, status, None)]
    if shape == "eventlog":
        ts = 1_700_000_000_000_000 + torch.cumsum(rnd(1, 2000), 0)
        tenants = torch.randint(1, 900_124, (8,), device=device, dtype=torch.int64, generator=g)
        other = torch.tensor([302, 404, 500], device=device, dtype=torch.int64)
        status = torch.where(torch.rand((n,), device=device, generator=g) < 0.97, torch.full_like(i, 200), other[rnd(0, 3)])
        return [(capi.OBJ_DATETIME, ts, None), (capi.OBJ_INT, tenants[rnd(0, 8)], None), (capi.OBJ_INT, status, None),
                (capi.OBJ_INT, 10**12 + rnd(0, 10**6), None), (capi.OBJ_INT, rnd(0, 1 << 20), None)]
    raise ValueError(f"shape {shape!r}: one of {ENCODE_SHAPES}")
