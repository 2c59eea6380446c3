"""Major-compaction merge: host mirror of include/obgpu_compaction.h plus the multi-GPU driver.

Reference: ObPartitionMajorMerger::merge_partition (compaction/ob_partition_merger.cpp:678-829) merges
the tables of a tablet by rowkey and fuses rows of one rowkey newest first; parallel merge cuts the
rowkey space into ranges at macro-block boundaries (ObParallelMergeCtx,
compaction/ob_partition_parallel_merge_ctx.cpp:187-424) and merges every range independently, the
outputs being concatenated in range order. The multi-GPU driver below does the same with one range
per rank: sample rowkeys -> all_gather -> pick world-1 splitters -> every rank sends the slice of each
run it owns to the rank owning that range (the one exchange step of the path, NCCL over NVLink) ->
local K-way merge on the device -> rank order is global rowkey order.

torch is used for device memory and torch.distributed only; the merge itself is libobgpu_scan.so.
"""
import ctypes as C
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from . import capi
from .capi import lib, check


@dataclass
class DecodedRun:
    """One sorted run as dense column tensors (device tensors for the GPU path)."""
    key: object                    # int64 [n]
    flag: Optional[object]         # uint8 [n] ObDmlFlag, or None = every row DF_INSERT
    vals: List[object]             # n_cols x int64 [n]
    ext: List[object]              # n_cols x uint8 [n]  (0 value, 1 NULL, 2 NOP)
    more_keys: Optional[List[object]] = None   # rowkey columns after the first (composite rowkeys), int64 [n] each

    @property
    def n(self):
        return int(self.key.shape[0])

    def slice(self, lo, hi):
        return DecodedRun(self.key[lo:hi], None if self.flag is None else self.flag[lo:hi],
                          [v[lo:hi] for v in self.vals], [e[lo:hi] for e in self.ext],
                          None if self.more_keys is None else [k[lo:hi] for k in self.more_keys])


def decode_run(ctx, table, key_col: int, flag_col: Optional[int], cols: Sequence[int], device=None,
               device_image_ptr: Optional[int] = None, batch=None, check_rowkey: bool = True) -> DecodedRun:
    """Opens `table` as a page batch on ctx (or takes an already open `batch`, which stays open) and decodes rowkey,
    flag and payload columns into torch tensors on the ctx device (obgpu_batch_decode_column)."""
    import torch
    device = device or torch.device("cuda", torch.cuda.current_device())
    own = batch is None
    if own:
        batch = ctx.open_batch(table, device_image_ptr=device_image_ptr)
    n = batch.total_rows

    all_cols = [key_col] + ([flag_col] if flag_col is not None else []) + list(cols)
    vs = [torch.empty(n, dtype=torch.int64, device=device) for _ in all_cols]
    es = [torch.empty(n, dtype=torch.uint8, device=device) for _ in all_cols]
    for k in range(0, len(all_cols), 16):   # one launch per 16 columns: every block image is read once
        sub = all_cols[k:k + 16]
        ci = (C.c_int32 * len(sub))(*sub)
        vp = (C.c_void_p * len(sub))(*[v.data_ptr() for v in vs[k:k + 16]])
        ep = (C.c_void_p * len(sub))(*[e.data_ptr() for e in es[k:k + 16]])
        check(lib.obgpu_batch_decode_columns(batch._h, len(sub), ci, vp, ep), "obgpu_batch_decode_columns", ctx._h)
    key, key_ext = vs[0], es[0]
    flag = None
    at = 1
    if flag_col is not None:
        flag = vs[1].to(torch.uint8)
        at = 2
    vals, ext = vs[at:], es[at:]
    if own:
        batch.close()
    if check_rowkey and bool((key_ext != 0).any()):
        raise capi.ObGpuError(capi.OB_INVALID_DATA, "decode_run", "rowkey column holds NULL / NOP cells")
    return DecodedRun(key, flag, vals, ext)


class MergeResult:
    def __init__(self, ctx, handle, n_cols, keep):
        self.ctx, self._h, self.n_cols, self._keep = ctx, handle, n_cols, keep

    def info(self) -> capi.MergeInfo:
        info = capi.MergeInfo()
        check(lib.obgpu_merge_result_info(self._h, C.byref(info)), "obgpu_merge_result_info", self.ctx._h)
        return info

    def fetch(self, col: int, row_begin=0, row_count=None):
        """(values int64, null bytes) of output column `col` (-1: rowkey) on the host."""
        n = self.info().out_rows
        if row_count is None:
            row_count = n - row_begin
        v = np.empty(row_count, dtype=np.int64)
        nl = np.empty(row_count, dtype=np.uint8)
        check(lib.obgpu_merge_result_fetch(self._h, col, row_begin, row_count, v.ctypes.data, nl.ctypes.data),
              "obgpu_merge_result_fetch", self.ctx._h)
        return v, nl

    def fetch_strings(self, col: int, row_begin=0, row_count=None):
        """String column `col` of the merged stream: (heap bytes uint8, offsets int64 [rows + 1], null bytes)."""
        n = self.info().out_rows
        if row_count is None:
            row_count = n - row_begin
        off = np.zeros(row_count + 1, dtype=np.int64)
        nl = np.zeros(max(row_count, 1), dtype=np.uint8)
        need = C.c_int64(0)
        code = lib.obgpu_merge_result_fetch_strings(self._h, col, row_begin, row_count, None, 0, off.ctypes.data,
                                                    nl.ctypes.data, C.byref(need))
        if code not in (capi.OB_SUCCESS, capi.OB_BUF_NOT_ENOUGH):
            check(code, "obgpu_merge_result_fetch_strings(size)", self.ctx._h)
        heap = np.zeros(max(need.value, 1), dtype=np.uint8)
        if need.value > 0:
            check(lib.obgpu_merge_result_fetch_strings(self._h, col, row_begin, row_count, heap.ctypes.data, heap.size,
                                                       off.ctypes.data, nl.ctypes.data, C.byref(need)),
                  "obgpu_merge_result_fetch_strings", self.ctx._h)
        return heap[:need.value], off, nl[:row_count]

    def set_string_images(self, device_ptrs: Sequence[int], sizes: Sequence[int]):
        arr = (C.c_void_p * max(len(device_ptrs), 1))(*device_ptrs)
        sz = np.ascontiguousarray(sizes, dtype=np.int64)
        check(lib.obgpu_merge_result_set_string_images(self._h, arr, sz.ctypes.data, len(device_ptrs)),
              "obgpu_merge_result_set_string_images", self.ctx._h)

    def free(self):
        if self._h and self.ctx._h:
            lib.obgpu_merge_result_free(self._h)
        self._h = C.c_void_p()
        self._keep = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def merge_decoded(ctx, runs: Sequence[DecodedRun], default_vals=None, default_null=None) -> MergeResult:
    """obgpu_merge_decoded over device-resident runs (runs[0] oldest ... runs[-1] newest)."""
    n_cols = len(runs[0].vals)
    arr = (capi.MergeRun * len(runs))()
    keep = []
    for i, r in enumerate(runs):
        assert len(r.vals) == n_cols and len(r.ext) == n_cols
        vp = (C.c_void_p * max(n_cols, 1))(*[v.data_ptr() for v in r.vals])
        ep = (C.c_void_p * max(n_cols, 1))(*[e.data_ptr() for e in r.ext])
        keep += [vp, ep, r]
        arr[i].n = r.n
        arr[i].key = r.key.data_ptr()
        arr[i].flag = r.flag.data_ptr() if r.flag is not None else None
        arr[i].vals = vp
        arr[i].ext = ep
        if r.more_keys:
            mp = (C.c_void_p * len(r.more_keys))(*[k.data_ptr() for k in r.more_keys])
            keep.append(mp)
            arr[i].more_keys = mp
            arr[i].n_more_keys = len(r.more_keys)
    dv = dn = None
    if default_vals is not None:
        dv = np.ascontiguousarray(default_vals, dtype=np.int64)
    if default_null is not None:
        dn = np.ascontiguousarray(default_null, dtype=np.uint8)
    h = C.c_void_p()
    check(lib.obgpu_merge_decoded(ctx._h, arr, len(runs), n_cols, dv.ctypes.data if dv is not None else None,
                                  dn.ctypes.data if dn is not None else None, C.byref(h)), "obgpu_merge_decoded", ctx._h)
    return MergeResult(ctx, h, n_cols, keep)


class Comm:
    """obgpu_comm: NCCL communicator bound inside the library (one process per GPU). The 128-byte id comes from rank 0
    (Comm.unique_id()) and reaches the other ranks through the caller's own channel -- torch.distributed here."""

    def __init__(self, ctx, comm_id: bytes, rank: int, world: int):
        self.ctx, self.rank, self.world = ctx, rank, world
        self._h = C.c_void_p()
        buf = C.create_string_buffer(bytes(comm_id), 128)
        check(lib.obgpu_comm_create(ctx._h, buf, rank, world, C.byref(self._h)), "obgpu_comm_create", ctx._h)

    @staticmethod
    def unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        check(lib.obgpu_comm_unique_id(buf), "obgpu_comm_unique_id")
        return bytes(buf.raw)

    @staticmethod
    def from_torch_distributed(ctx, device=None, group=None) -> "Comm":
        """Rank 0 makes the id, a broadcast hands it out."""
        import torch
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        device = device or torch.device("cuda", torch.cuda.current_device())
        t = torch.zeros(128, dtype=torch.uint8, device=device)
        if rank == 0:
            t.copy_(torch.frombuffer(bytearray(Comm.unique_id()), dtype=torch.uint8))
        dist.broadcast(t, src=0 if group is None else dist.get_global_rank(group, 0), group=group)
        return Comm(ctx, bytes(t.cpu().numpy().tobytes()), rank, world)

    def close(self):
        if self._h:
            lib.obgpu_comm_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def merge_decoded_distributed(ctx, comm: Comm, local_runs: Dict[int, DecodedRun], n_runs_total: int, n_cols: int,
                              n_more_keys: int = 0, default_vals=None, default_null=None, samples_per_run: int = 1024):
    """obgpu_merge_decoded_distributed: the range-partitioned merge with the exchange inside the library (NCCL on the ctx
    stream). Returns (MergeResult of this rank's rowkey range, splitters, rows received per run)."""
    idx = sorted(local_runs)
    arr = (capi.MergeRun * max(len(idx), 1))()
    keep = []
    for i, q in enumerate(idx):
        r = local_runs[q]
        vp = (C.c_void_p * max(n_cols, 1))(*[v.data_ptr() for v in r.vals])
        ep = (C.c_void_p * max(n_cols, 1))(*[e.data_ptr() for e in r.ext])
        keep += [vp, ep, r]
        arr[i].n = r.n
        arr[i].key = r.key.data_ptr()
        arr[i].flag = r.flag.data_ptr() if r.flag is not None else None
        arr[i].vals, arr[i].ext = vp, ep
        if n_more_keys:
            mp = (C.c_void_p * n_more_keys)(*[k.data_ptr() for k in r.more_keys])
            keep.append(mp)
            arr[i].more_keys = mp
        arr[i].n_more_keys = n_more_keys
    ri = (C.c_int32 * max(len(idx), 1))(*idx)
    dv = np.ascontiguousarray(default_vals, dtype=np.int64) if default_vals is not None else None
    dn = np.ascontiguousarray(default_null, dtype=np.uint8) if default_null is not None else None
    split = np.zeros(max(comm.world - 1, 1), dtype=np.int64)
    recv = np.zeros(n_runs_total, dtype=np.int64)
    h = C.c_void_p()
    check(lib.obgpu_merge_decoded_distributed(ctx._h, comm._h, arr, ri, len(idx), n_runs_total, n_cols, n_more_keys,
                                              dv.ctypes.data if dv is not None else None,
                                              dn.ctypes.data if dn is not None else None, samples_per_run, C.byref(h),
                                              split.ctypes.data, recv.ctypes.data), "obgpu_merge_decoded_distributed", ctx._h)
    return MergeResult(ctx, h, n_cols, keep), split[:comm.world - 1], recv


def merge_batches(ctx, batches, rowkey_col, flag_col: Optional[int], cols: Sequence[int], default_vals=None,
                  default_null=None) -> MergeResult:
    """obgpu_merge_runs(_keys): the whole merge of one range from opened page batches (oldest first). rowkey_col: one
    column index or the list of a composite rowkey. String payload columns travel as references into the batches, which
    must stay open until the strings have been fetched."""
    arr = (C.c_void_p * len(batches))(*[b._h for b in batches])
    ci = (C.c_int32 * max(len(cols), 1))(*cols)
    if not isinstance(rowkey_col, int):
        keys = list(rowkey_col)
        kc = (C.c_int32 * len(keys))(*keys)
        dv = np.ascontiguousarray(default_vals, dtype=np.int64) if default_vals is not None else None
        dn = np.ascontiguousarray(default_null, dtype=np.uint8) if default_null is not None else None
        h = C.c_void_p()
        check(lib.obgpu_merge_runs_keys(ctx._h, arr, len(batches), kc, len(keys), -1 if flag_col is None else flag_col, ci,
                                        len(cols), dv.ctypes.data if dv is not None else None,
                                        dn.ctypes.data if dn is not None else None, C.byref(h)), "obgpu_merge_runs_keys", ctx._h)
        return MergeResult(ctx, h, len(cols), list(batches))
    dv = np.ascontiguousarray(default_vals, dtype=np.int64) if default_vals is not None else None
    dn = np.ascontiguousarray(default_null, dtype=np.uint8) if default_null is not None else None
    h = C.c_void_p()
    check(lib.obgpu_merge_runs(ctx._h, arr, len(batches), rowkey_col, -1 if flag_col is None else flag_col, ci, len(cols),
                               dv.ctypes.data if dv is not None else None, dn.ctypes.data if dn is not None else None,
                               C.byref(h)), "obgpu_merge_runs", ctx._h)
    return MergeResult(ctx, h, len(cols), list(batches))


def write_merged_sstable(res: MergeResult, rows_per_block: int = 1400, payload_encoding=None, n_threads: int = 0,
                         string_cols: Sequence[int] = ()):
    """The merged row stream as a new major SSTable shard (ObMacroBlockWriter::append_row ->
    ObMicroBlockEncoder::build_block in the reference, blocksstable/ob_macro_block_writer.cpp:837): rowkey
    INTEGER_BASE_DIFF, payload RAW unless told otherwise; every row DF_INSERT, so no flag column and no NOP.
    The encoder runs on the host (it does in the reference too); the block bytes are reference-format."""
    from .sstable import Column, encode_table
    key, _ = res.fetch(-1)
    cols = [Column(capi.OBJ_INT, capi.ENC_INTEGER_BASE_DIFF, key)]
    for c in range(res.n_cols):
        enc = capi.ENC_RAW if payload_encoding is None else payload_encoding[c]
        if c in string_cols:
            heap, off, nl = res.fetch_strings(c)
            cols.append(Column(capi.OBJ_VARCHAR, enc, None, nulls=nl if nl.any() else None, str_heap=heap, str_off=off))
        else:
            v, nl = res.fetch(c)
            cols.append(Column(capi.OBJ_INT, enc, v, nulls=nl if nl.any() else None))
    return encode_table(cols, rows_per_block, rowkey_cnt=1, n_threads=n_threads)


# ---- phase B on the device: merged columns -> SSTable bytes + column checksums -------------------------------------------
class Encoded:
    """Device-encoded micro-blocks (obgpu_encoded): PAX blocks, byte for byte what the host writer produces for the same rows
    and per-column encodings (ObMicroBlockEncoder::build_block; RAW on every column unless encodings were given). A block of
    size 0 is left to the host writer (info().n_host_blocks counts them)."""

    def __init__(self, ctx, handle, n_cols, keep=None):
        self.ctx, self._h, self.n_cols, self._keep = ctx, handle, n_cols, keep

    def info(self) -> capi.EncodedInfo:
        info = capi.EncodedInfo()
        check(lib.obgpu_encoded_get_info(self._h, C.byref(info)), "obgpu_encoded_get_info", self.ctx._h)
        return info

    def fetch(self):
        """(image uint8, offsets int64, sizes int64); a size of 0 marks a block left to the host writer."""
        info = self.info()
        img = np.zeros(max(info.image_size, 1), dtype=np.uint8)
        off = np.zeros(info.n_blocks, dtype=np.int64)
        sz = np.zeros(info.n_blocks, dtype=np.int64)
        check(lib.obgpu_encoded_fetch(self._h, img.ctypes.data, img.size, off.ctypes.data, sz.ctypes.data, info.n_blocks),
              "obgpu_encoded_fetch", self.ctx._h)
        return img[:info.image_size], off, sz

    def device_image(self):
        """(device pointer of the image, of the int64 offsets, of the uint32 sizes) -- valid until free()."""
        a, b, c = C.c_void_p(), C.c_void_p(), C.c_void_p()
        check(lib.obgpu_encoded_device_image(self._h, C.byref(a), C.byref(b), C.byref(c)), "obgpu_encoded_device_image", self.ctx._h)
        return a.value, b.value, c.value

    def column_checksums(self) -> np.ndarray:
        out = np.zeros(self.n_cols, dtype=np.int64)
        check(lib.obgpu_encoded_column_checksums(self._h, out.ctypes.data), "obgpu_encoded_column_checksums", self.ctx._h)
        return out

    def free(self):
        if self._h and self.ctx._h:
            lib.obgpu_encoded_free(self._h)
        self._h = C.c_void_p()
        self._keep = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _encode_cols(cols):
    arr = (capi.EncodeCol * len(cols))()
    for i, (vals_ptr, null_ptr, obj_type, byte_only) in enumerate(cols):
        arr[i].dev_vals = vals_ptr
        arr[i].dev_null = null_ptr
        arr[i].obj_type = obj_type
        arr[i].byte_packing_only = 1 if byte_only else 0
    return arr


DEVICE_ENCODINGS = (capi.ENC_RAW, capi.ENC_DICT, capi.ENC_RLE, capi.ENC_CONST, capi.ENC_INTEGER_BASE_DIFF, capi.ENC_AUTO)


def _encodings(encodings, n_cols) -> np.ndarray:
    """encodings -> int32 array of n_cols codecs the device encoder takes (RAW / DICT / RLE / CONST / INTEGER_BASE_DIFF / AUTO)."""
    enc = np.ascontiguousarray(encodings, dtype=np.int32)
    if enc.shape != (n_cols,):
        raise ValueError(f"encodings: {n_cols} values expected, got {enc.size}")
    bad = [int(e) for e in enc if int(e) not in DEVICE_ENCODINGS]
    if bad:
        raise ValueError(f"encodings: {bad} not among the device encoder's codecs {DEVICE_ENCODINGS}")
    return enc


def encode_columns(ctx, cols, total_rows: int, rows_per_block: int, rowkey_cnt: int = 0, align: int = 128, keep=None,
                   encodings: Optional[Sequence[int]] = None) -> Encoded:
    """cols: (device pointer of the int64 value images, device pointer of the NULL bytes or None, OBJ_* type, byte_packing_only).
    encodings: one ENC_RAW / ENC_DICT / ENC_RLE / ENC_CONST / ENC_INTEGER_BASE_DIFF / ENC_AUTO per column (None: every column RAW)."""
    h = C.c_void_p()
    if encodings is not None:
        enc = _encodings(encodings, len(cols))
    arr = _encode_cols(cols)
    if encodings is None:
        check(lib.obgpu_encode_columns(ctx._h, arr, len(cols), rowkey_cnt, total_rows, rows_per_block, align, C.byref(h)),
              "obgpu_encode_columns", ctx._h)
    else:
        check(lib.obgpu_encode_columns_with(ctx._h, arr, enc.ctypes.data, len(cols), rowkey_cnt, total_rows, rows_per_block, align,
                                            C.byref(h)), "obgpu_encode_columns_with", ctx._h)
    return Encoded(ctx, h, len(cols), keep)


def column_checksums(ctx, cols, total_rows: int) -> np.ndarray:
    out = np.zeros(len(cols), dtype=np.int64)
    arr = _encode_cols(cols)
    check(lib.obgpu_column_checksums(ctx._h, arr, len(cols), total_rows, out.ctypes.data), "obgpu_column_checksums", ctx._h)
    return out


def encode_merge_result(res: MergeResult, result_cols: Sequence[int], obj_types: Sequence[int], rows_per_block: int,
                        rowkey_cnt: int = 1, align: int = 128, encodings: Optional[Sequence[int]] = None) -> Encoded:
    """One column group of the merged stream (-1: the rowkey, -2 ...: further rowkey columns, >= 0 payload columns).
    encodings: one codec per column as in encode_columns (None: every column RAW)."""
    rc = np.ascontiguousarray(result_cols, dtype=np.int32)
    ot = np.ascontiguousarray(obj_types, dtype=np.int32)
    h = C.c_void_p()
    if encodings is None:
        check(lib.obgpu_merge_result_encode(res._h, rc.ctypes.data, ot.ctypes.data, len(rc), rowkey_cnt, rows_per_block, align,
                                            C.byref(h)), "obgpu_merge_result_encode", res.ctx._h)
    else:
        enc = _encodings(encodings, len(rc))
        check(lib.obgpu_merge_result_encode_with(res._h, rc.ctypes.data, ot.ctypes.data, enc.ctypes.data, len(rc), rowkey_cnt,
                                                 rows_per_block, align, C.byref(h)), "obgpu_merge_result_encode_with", res.ctx._h)
    return Encoded(res.ctx, h, len(rc), res)


def co_merge_write(res: MergeResult, column_groups: Sequence[Sequence[int]], obj_types: Dict[int, int], rows_per_block: int,
                   align: int = 128, encodings: Optional[Dict[int, int]] = None) -> List[Encoded]:
    """Column-oriented merge, writer side (ObCOMergeLogReplayer::replay_merge_log -> ObCOMergeWriter -> ObWriteHelper::project /
    append, column_store/ob_column_oriented_merger.cpp:722-745, ob_co_merge_writer.cpp:67-117): the merged stream is produced
    ONCE and replayed into the writer of every column group; here every group is one obgpu_merge_result_encode over the columns
    the group projects. A group that holds the rowkey (-1 first) is written with rowkey_cnt 1, a pure column group with 0.
    encodings: column -> codec (as encode_columns takes them; a column it does not name is RAW); None: every column RAW."""
    out = []
    for cg in column_groups:
        cg = list(cg)
        rk = 1 if cg and cg[0] == -1 else 0
        enc = None if encodings is None else [encodings.get(c, capi.ENC_RAW) for c in cg]
        out.append(encode_merge_result(res, cg, [obj_types[c] for c in cg], rows_per_block, rowkey_cnt=rk, align=align, encodings=enc))
    return out


# ---- multi-GPU: range partition + one exchange step ----------------------------------------------------
# ---- runs larger than device memory: range by range, copies of the next range under the merge of this one ---------------------
def streamed_major_merge(tables: Sequence[object], end_keys: Sequence[np.ndarray], key_col: int,
                         flag_col: Optional[int], cols: Sequence[int], n_ranges: int, sink: Callable[[int, "MergeResult"], None],
                         device=None, default_vals=None, default_null=None, n_workers: int = 2):
    """Major merge of runs that do not fit in device memory together (ObPartitionMajorMerger over a tablet whose tables exceed HBM).
    tables[q]: the run's SSTable in HOST memory (oldest first); end_keys[q][b]: last rowkey of its micro-block b (the index rows).
    The rowkey space is cut into n_ranges ranges at quantiles of the block end keys (the reference cuts parallel-merge ranges at
    macro-block boundaries the same way, ob_partition_parallel_merge_ctx.cpp:187-424). A range is one unit of work: the micro-blocks
    of every run that can hold its rowkeys are opened as a page batch straight from host memory (the host->device copy), decoded,
    cut to the range with a binary search on the decoded rowkeys, merged, and handed to sink(range_index, MergeResult) (which
    fetches / encodes the rows: the device->host side). n_workers ranges are in flight, each on its own ctx / stream, so the copies
    of range i + 1 run under the merge and the fetch of range i; device memory holds n_workers ranges at a time.
    Ranges come back in order: sink is called with 0, 1, 2 ... (rowkey order of the whole output)."""
    import threading
    import torch
    from .sstable import TableImage
    device = device or torch.device("cuda", torch.cuda.current_device())
    allk = np.sort(np.concatenate([np.asarray(e, dtype=np.int64) for e in end_keys]))
    cuts = [int(allk[min(len(allk) - 1, (len(allk) * (i + 1)) // n_ranges)]) for i in range(n_ranges - 1)]
    cuts = sorted(set(cuts))
    bounds = [None] + cuts + [None]          # range i = (bounds[i], bounds[i + 1]]  (None: open)
    n_ranges = len(bounds) - 1
    results = [None] * n_ranges
    errors = []
    done = [threading.Event() for _ in range(n_ranges)]
    next_range = [0]
    lock = threading.Lock()

    def work():
        from .scan import ScanContext
        torch.cuda.set_device(device)
        stream = torch.cuda.Stream(device=device)          # this worker's stream: torch tensors and the library's launches share it
        ctx = ScanContext(device.index if device.index is not None else 0, stream=stream.cuda_stream)
        try:
            while True:
                with lock:
                    i = next_range[0]
                    next_range[0] += 1
                if i >= n_ranges:
                    break
                lo, hi = bounds[i], bounds[i + 1]
                runs = []
                with torch.cuda.stream(stream):
                    for q, tb in enumerate(tables):
                        ek = np.asarray(end_keys[q], dtype=np.int64)
                        b0 = 0 if lo is None else int(np.searchsorted(ek, lo, side="right"))     # first block whose last key > lo
                        b1 = len(ek) if hi is None else min(len(ek), int(np.searchsorted(ek, hi, side="left")) + 1)
                        if b0 >= b1:
                            runs.append(DecodedRun(torch.empty(0, dtype=torch.int64, device=device), None if flag_col is None else
                                                   torch.empty(0, dtype=torch.uint8, device=device),
                                                   [torch.empty(0, dtype=torch.int64, device=device) for _ in cols],
                                                   [torch.empty(0, dtype=torch.uint8, device=device) for _ in cols]))
                            continue
                        o0 = int(tb.offsets[b0])
                        o1 = int(tb.offsets[b1 - 1]) + int(tb.sizes[b1 - 1])
                        sub = TableImage(tb.image[o0:o1], np.asarray(tb.offsets[b0:b1]) - o0, tb.sizes[b0:b1], 0, tb.n_cols)
                        d = decode_run(ctx, sub, key_col, flag_col, cols, device=device)
                        ctx.synchronize()
                        r0 = 0 if lo is None else int(torch.searchsorted(d.key, torch.tensor([lo], device=device), right=True)[0])
                        r1 = d.n if hi is None else int(torch.searchsorted(d.key, torch.tensor([hi], device=device), right=True)[0])
                        runs.append(d.slice(r0, r1))
                    res = merge_decoded(ctx, runs, default_vals, default_null)
                    res.info()
                # hand the ranges over in order
                if i > 0:
                    done[i - 1].wait()
                if not errors:
                    sink(i, res)
                res.free()
                del runs
                done[i].set()
        except Exception as e:   # pragma: no cover
            errors.append(e)
            for ev in done:
                ev.set()
        finally:
            ctx.close()

    threads = [threading.Thread(target=work) for _ in range(max(1, n_workers))]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    return n_ranges


def merge_runs_streamed(device: int, tables: Sequence[object], end_keys: Sequence[np.ndarray], key_col: int, flag_col: Optional[int],
                        cols: Sequence[int], n_ranges: int, sink: Callable[[int, "MergeResult"], None], n_streams: int = 2,
                        default_vals=None, default_null=None) -> int:
    """obgpu_merge_runs_streamed: the range loop of streamed_major_merge inside the library (worker threads, one ctx / stream each).
    sink(range_index, MergeResult) is called in rowkey order; the result is only valid inside the call."""
    arr = (capi.StreamRun * len(tables))()
    keep = []
    for q, tb in enumerate(tables):
        offs = np.ascontiguousarray(tb.offsets, dtype=np.int64)
        sizes = np.ascontiguousarray(tb.sizes, dtype=np.int64)
        ek = np.ascontiguousarray(end_keys[q], dtype=np.int64)
        keep += [offs, sizes, ek]
        arr[q].image, arr[q].offsets, arr[q].sizes, arr[q].end_keys = tb.image.ctypes.data, offs.ctypes.data, sizes.ctypes.data, ek.ctypes.data
        arr[q].n_blocks = len(offs)
    ci = (C.c_int32 * max(len(cols), 1))(*cols)
    dv = None if default_vals is None else np.ascontiguousarray(default_vals, dtype=np.int64)
    dn = None if default_null is None else np.ascontiguousarray(default_null, dtype=np.uint8)
    errors = []

    class _Ctx:   # the result's ctx is the worker's: only what MergeResult.fetch needs
        _h = None

    def cb(_arg, rng, res_h):
        try:
            r = MergeResult(_Ctx, C.c_void_p(res_h), len(cols), None)
            sink(int(rng), r)
            r._h = C.c_void_p()     # owned by the library
            return capi.OB_SUCCESS
        except Exception as e:      # pragma: no cover
            errors.append(e)
            return capi.OB_ERR_SYS

    cfn = capi.MERGE_SINK(cb)
    done = C.c_int32(0)
    code = lib.obgpu_merge_runs_streamed(device, n_streams, arr, len(tables), key_col, -1 if flag_col is None else flag_col, ci, len(cols),
                                        dv.ctypes.data if dv is not None else None, dn.ctypes.data if dn is not None else None,
                                        n_ranges, cfn, None, C.byref(done))
    if errors:
        raise errors[0]
    if code != capi.OB_SUCCESS:
        raise capi.ObGpuError(code, "obgpu_merge_runs_streamed", "")
    return done.value


def choose_splitters(candidates, world: int):
    """world-1 splitters at the quantiles of the gathered rowkey samples (sorted, duplicates kept)."""
    import torch
    c, _ = torch.sort(candidates)
    if world <= 1 or c.numel() == 0:
        return c[:0]
    idx = (torch.arange(1, world, device=c.device, dtype=torch.int64) * c.numel()) // world
    return c[idx.clamp(max=c.numel() - 1)]


def _pack(run: DecodedRun, lo: int, hi: int):
    """One contiguous byte buffer per (run, destination): int64 sections first (alignment), then bytes."""
    import torch
    n = hi - lo
    n_cols = len(run.vals)
    more = run.more_keys or []
    n64 = 1 + n_cols + len(more)               # rowkey, payload, then the remaining rowkey columns of a composite rowkey
    buf = torch.empty(n * (8 * n64 + 1 + n_cols), dtype=torch.uint8, device=run.key.device)
    i64 = buf[:8 * n * n64].view(torch.int64)
    i64[:n] = run.key[lo:hi]
    for c in range(n_cols):
        i64[(1 + c) * n:(2 + c) * n] = run.vals[c][lo:hi]
    for c, k in enumerate(more):
        i64[(1 + n_cols + c) * n:(2 + n_cols + c) * n] = k[lo:hi]
    b = buf[8 * n * n64:]
    if run.flag is None:
        b[:n] = capi.DF_INSERT
    else:
        b[:n] = run.flag[lo:hi]
    for c in range(n_cols):
        b[(1 + c) * n:(2 + c) * n] = run.ext[c][lo:hi]
    return buf


def _unpack(buf, n: int, n_cols: int, n_more: int = 0) -> DecodedRun:
    import torch
    n64 = 1 + n_cols + n_more
    i64 = buf[:8 * n * n64].view(torch.int64)
    b = buf[8 * n * n64:]
    return DecodedRun(i64[:n], b[:n], [i64[(1 + c) * n:(2 + c) * n] for c in range(n_cols)],
                      [b[(1 + c) * n:(2 + c) * n] for c in range(n_cols)],
                      [i64[(1 + n_cols + c) * n:(2 + n_cols + c) * n] for c in range(n_more)] if n_more else None)


def distributed_major_merge(local_runs: Dict[int, DecodedRun], n_runs_total: int, n_cols: int,
                            merge_fn: Callable[[List[DecodedRun]], object], group=None, samples_per_run: int = 1024):
    """Range-partitioned merge over the ranks of `group`.

    local_runs: run index -> DecodedRun for the runs this rank holds (every run index in
    [0, n_runs_total) is held by exactly one rank). merge_fn merges a list of DecodedRun ordered oldest
    -> newest and returns whatever the caller wants back (the GPU path passes merge_decoded).
    Returns (merge_fn result for this rank's rowkey range, splitters, received row counts)."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    some = next(iter(local_runs.values())) if local_runs else None
    device = some.key.device if some is not None else torch.device("cpu")
    # 1. candidates: evenly spaced rowkeys of every local run; padded with the maximum so that the gather is rectangular
    per_rank_slots = samples_per_run * n_runs_total
    cand = torch.full((per_rank_slots,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=device)
    valid = torch.zeros((), dtype=torch.int64, device=device)
    at = 0
    for q in sorted(local_runs):
        r = local_runs[q]
        if r.n == 0:
            continue
        k = min(samples_per_run, r.n)
        idx = (torch.arange(k, device=device, dtype=torch.int64) * r.n) // k
        cand[at:at + k] = r.key[idx]
        at += k
    valid += at
    if world > 1:
        gathered = [torch.empty_like(cand) for _ in range(world)]
        dist.all_gather(gathered, cand, group=group)
        counts = [torch.empty_like(valid) for _ in range(world)]
        dist.all_gather(counts, valid, group=group)
        allc = torch.cat([g[:int(c)] for g, c in zip(gathered, counts)])
    else:
        allc = cand[:at]
    splitters = choose_splitters(allc, world)
    # 2. slice boundaries of every local run, row-count matrix [run, destination]
    bounds = {}
    cnt = torch.zeros((n_runs_total, world), dtype=torch.int64, device=device)
    for q, r in local_runs.items():
        b = torch.searchsorted(r.key.contiguous(), splitters, right=False) if world > 1 else splitters.new_zeros(0)
        b = [0] + [int(x) for x in b.tolist()] + [r.n]
        bounds[q] = b
        cnt[q] = torch.tensor([b[j + 1] - b[j] for j in range(world)], dtype=torch.int64, device=device)
    owner = torch.full((n_runs_total,), -1, dtype=torch.int64, device=device)
    for q in local_runs:
        owner[q] = rank
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)      # every row of cnt is filled by exactly one rank
        dist.all_reduce(owner, op=dist.ReduceOp.MAX, group=group)
    cnt_h = cnt.cpu().numpy()
    owner_h = owner.cpu().numpy()
    if (owner_h < 0).any():
        raise ValueError("every run index must be held by exactly one rank")
    # 3. the exchange: one packed buffer per (run, destination)
    recv = {}
    ops, keep = [], []
    # composite rowkeys: the partition looks at the first rowkey column only (rows that tie on it stay on one rank), the
    # other rowkey columns travel like payload; every rank must agree on their number
    n_more_t = torch.tensor([len(some.more_keys or []) if some is not None else 0], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(n_more_t, op=dist.ReduceOp.MAX, group=group)
    n_more = int(n_more_t.item())
    row_bytes = 8 * (1 + n_cols + n_more) + 1 + n_cols
    for q in range(n_runs_total):
        o = int(owner_h[q])
        if o == rank:
            b = bounds[q]
            for j in range(world):
                n = b[j + 1] - b[j]
                if j == rank:
                    recv[q] = local_runs[q].slice(b[j], b[j + 1])
                elif n > 0:
                    buf = _pack(local_runs[q], b[j], b[j + 1])
                    keep.append(buf)
                    ops.append(dist.P2POp(dist.isend, buf, j if group is None else dist.get_global_rank(group, j), group))
        else:
            n = int(cnt_h[q][rank])
            if n > 0:
                buf = torch.empty(n * row_bytes, dtype=torch.uint8, device=device)
                recv[q] = (buf, n)
                ops.append(dist.P2POp(dist.irecv, buf, o if group is None else dist.get_global_rank(group, o), group))
            else:
                recv[q] = None
    if ops:
        for w in dist.batch_isend_irecv(ops):
            w.wait()
    runs = []
    for q in range(n_runs_total):
        x = recv.get(q)
        if x is None:
            z = torch.zeros(0, dtype=torch.int64, device=device)
            zb = torch.zeros(0, dtype=torch.uint8, device=device)
            runs.append(DecodedRun(z, zb, [z] * n_cols, [zb] * n_cols, [z] * n_more if n_more else None))
        elif isinstance(x, tuple):
            runs.append(_unpack(x[0], x[1], n_cols, n_more))
        else:
            runs.append(x)
    if device.type == "cuda":
        torch.cuda.current_stream(device).synchronize()  # the merge runs on the ctx stream
    return merge_fn(runs), splitters, cnt_h[:, rank].copy()
