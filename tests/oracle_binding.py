"""ctypes binding of the CPU oracle (oracle/libob_oracle.so). TEST INFRASTRUCTURE: only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_LIB = os.path.join(ORACLE_DIR, "libob_oracle.so")
REF_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_bitstream.so")
REF_CODEC_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_codec.so")
REF_BITMAP_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_bitmap.so")
REF_MISC_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_misc.so")
REF_MACRO_LIB = os.path.join(ORACLE_DIR, "_ref", "libref_macro.so")


def _cpu_stamp():
    """-march=native code must run where it was compiled: identify the host by its cpu flags."""
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    import hashlib
                    return hashlib.sha1(line.encode()).hexdigest()
    except OSError:
        pass
    return "unknown"


def build_oracle():
    global ORACLE_LIB
    if os.path.dirname(ORACLE_LIB) != ORACLE_DIR:   # already built for this host in a temporary directory
        return ORACLE_LIB
    src = [os.path.join(ORACLE_DIR, f) for f in ("ob_oracle.c", "ob_stream_codecs.c", "ob_oracle.h", "Makefile")]
    stamp_file = os.path.join(ORACLE_DIR, ".built_on")
    stamp = _cpu_stamp()
    try:
        with open(stamp_file) as f:
            same_host = f.read().strip() == stamp
    except OSError:
        same_host = False
    stale = (not os.path.exists(ORACLE_LIB)) or not same_host or \
        any(os.path.getmtime(s) > os.path.getmtime(ORACLE_LIB) for s in src)
    if stale and not os.access(ORACLE_DIR, os.W_OK):   # read-only tree: this host's build goes to a temporary directory
        out = tempfile.mkdtemp(prefix="ob_oracle_") + os.sep
        atexit.register(shutil.rmtree, out, True)
        subprocess.run(["make", "-B", "-C", ORACLE_DIR, "-s", "OUT=" + out, out + "libob_oracle.so"], check=True, capture_output=True)
        ORACLE_LIB = out + "libob_oracle.so"
    elif stale:
        subprocess.run(["make", "-B", "-C", ORACLE_DIR, "-s", "all"], check=True, capture_output=True)
        with open(stamp_file, "w") as f:
            f.write(stamp + "\n")
    elif os.path.isdir("/root/reference") and not (os.path.exists(REF_LIB) and os.path.exists(REF_CODEC_LIB) and os.path.exists(REF_BITMAP_LIB) and os.path.exists(REF_MISC_LIB) and os.path.exists(REF_MACRO_LIB)):
        subprocess.run(["make", "-C", ORACLE_DIR, "-s", "ref"], check=True, capture_output=True)
    return ORACLE_LIB


class OraParam(C.Structure):
    _fields_ = [("i64", C.c_int64), ("ptr", C.c_char_p), ("len", C.c_uint32), ("is_null", C.c_int32)]


class OraNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("op", C.c_int32), ("col", C.c_int32), ("param_begin", C.c_int32),
                ("n_params", C.c_int32), ("n_children", C.c_int32)]


class OraFilter(C.Structure):
    _fields_ = [("nodes", C.POINTER(OraNode)), ("n_nodes", C.c_int32), ("params", C.POINTER(OraParam)),
                ("n_params", C.c_int32)]


class OraDatum(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("len", C.c_uint32), ("is_null", C.c_int32), ("ival", C.c_uint64)]


class OraBlock(C.Structure):
    _fields_ = [("buf", C.c_void_p), ("size", C.c_int64), ("header_size", C.c_uint32), ("row_count", C.c_uint32),
                ("row_data_offset", C.c_uint32), ("column_count", C.c_uint16), ("rowkey_column_count", C.c_uint16),
                ("var_column_count", C.c_uint16), ("row_index_byte", C.c_uint8), ("extend_value_bit", C.c_uint8),
                ("col_headers", C.c_void_p), ("meta", C.c_void_p), ("row_data", C.c_void_p),
                ("row_data_len", C.c_int64),
                ("row_store_type", C.c_uint8), ("cs_off_width", C.c_uint8), ("cs_stream_count", C.c_uint16),
                ("cs_col_headers", C.c_void_p), ("cs_off_data", C.c_void_p), ("cs_first_stream_begin", C.c_uint32),
                ("cs_all_string_offset", C.c_uint32)]


class OraScanOut(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_void_p)), ("lens", C.POINTER(C.c_void_p)), ("nulls", C.POINTER(C.c_void_p)),
                ("has_null", C.c_void_p), ("row_ids", C.c_void_p), ("sel_offset", C.c_void_p),
                ("cap_rows", C.c_int64), ("string_base", C.c_uint64)]


_lib = None


class OraMergeRun(C.Structure):
    _fields_ = [("n", C.c_int64), ("key", C.c_void_p), ("flag", C.c_void_p), ("vals", C.POINTER(C.c_void_p)),
                ("ext", C.POINTER(C.c_void_p)), ("more_keys", C.POINTER(C.c_void_p)), ("n_more_keys", C.c_int32)]


def oracle():
    global _lib
    if _lib is None:
        build_oracle()
        L = C.CDLL(ORACLE_LIB)
        vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
        P = C.POINTER
        L.ora_bs_get.restype = u64
        L.ora_bs_get.argtypes = [vp, i64, i64]
        L.ora_bs_get_fast.restype = u64
        L.ora_bs_get_fast.argtypes = [vp, i64, i64, i64]
        L.ora_bs_set.restype = None
        L.ora_bs_set.argtypes = [vp, i64, i64, u64]
        L.ora_block_init.argtypes = [P(OraBlock), vp, i64]
        L.ora_block_verify_checksums.argtypes = [P(OraBlock)]
        L.ora_decode_cell.argtypes = [P(OraBlock), i32, i64, P(OraDatum)]
        L.ora_crc64_sse42.restype = u64
        L.ora_crc64_sse42.argtypes = [u64, vp, i64]
        L.ora_column_checksum.restype = i64
        L.ora_column_checksum.argtypes = [vp, vp, i64, i32]
        for f in ("ora_int_array_lower_bound", "ora_int_array_upper_bound"):
            getattr(L, f).restype = i64
            getattr(L, f).argtypes = [vp, i64, i64, i64, i64]
        L.ora_bitset_get_ref.restype = i64
        L.ora_bitset_get_ref.argtypes = [vp, i64]
        L.ora_arena_reset.restype = None
        L.ora_arena_reset.argtypes = []
        L.ora_dict_count.argtypes = [P(OraBlock), i32, P(i64)]
        L.ora_dict_entry.argtypes = [P(OraBlock), i32, i64, P(OraDatum)]
        L.ora_dict_refs.argtypes = [P(OraBlock), i32, C.c_void_p, i64, C.c_void_p]
        L.ora_get_rows_fixed.argtypes = [P(OraBlock), i32, vp, i64, i64, vp, i32, vp, P(i32)]
        L.ora_get_rows_discrete.argtypes = [P(OraBlock), i32, vp, i64, i64, vp, vp, vp, P(i32)]
        L.ora_filter_white.argtypes = [P(OraBlock), i32, i32, P(OraParam), i32, i64, i64, vp]
        L.ora_filter_tree.argtypes = [P(OraBlock), P(OraFilter), i64, i64, vp]
        L.ora_bitmap_get_row_ids.argtypes = [vp, i64, vp, P(i64), P(i64), i64, i64, i64]
        L.ora_bitmap_popcnt.restype = i64
        L.ora_bitmap_popcnt.argtypes = [vp, i64]
        L.ora_scan_blocks.argtypes = [vp, vp, vp, i32, i32, P(OraFilter), vp, i32, i32, i64, P(OraScanOut), P(i64),
                                      P(i64)]
        L.ora_scan_blocks_mt.argtypes = [vp, vp, vp, i32, P(OraFilter), vp, i32, i32, i32, P(i64), P(i64), P(u64)]
        L.ora_decode_column_ext.argtypes = [vp, vp, vp, i32, i32, vp, vp, i64, P(i64)]
        L.ora_major_merge.argtypes = [P(OraMergeRun), i32, i32, vp, vp, i64, vp, P(vp), P(vp), P(i64), P(i64)]
        L.ora_major_merge_keys.argtypes = [P(OraMergeRun), i32, i32, vp, vp, i64, vp, P(vp), P(vp), P(vp), P(i64), P(i64)]
        L.ora_agg_row_read.argtypes = [vp, i64, C.c_uint32, i32, P(vp), P(i32), P(i32)]
        L.ora_skip_index_filter.argtypes = [vp, i64, i64, vp, i32, P(OraFilter), P(i32)]
        _lib = L
    return _lib


def ref_bitstream():
    """The REAL reference ObBitStream (oracle/_ref), or None when it was never built."""
    if not os.path.exists(REF_LIB):
        return None
    L = C.CDLL(REF_LIB)
    L.ref_bs_get.restype = C.c_uint64
    L.ref_bs_get.argtypes = [C.c_void_p, C.c_int64, C.c_int64]
    L.ref_bs_get_unpack.restype = C.c_uint64
    L.ref_bs_get_unpack.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64]
    L.ref_bs_memory_safe_set.restype = None
    L.ref_bs_memory_safe_set.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_uint64]
    L.ref_bs_set.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int64]
    L.ref_bs_get_mask.restype = C.c_uint64
    L.ref_bs_get_mask.argtypes = [C.c_int64]
    return L


def ora_check(code, what):
    if code != 0:
        raise RuntimeError(f"oracle {what} failed: {code}")


def ora_flatten_filter(expr):
    """The checker's own post-order flattening of a filter tree (root last) into the oracle's structs. The expression
    objects are duck-typed (a leaf has .col / .op / .params, a logic node has .children and a class name of And / Or):
    nothing of the product's filter code runs on the oracle's side."""
    if expr is None:
        return None, None
    nodes, params, keep = [], [], []

    def visit(e):
        if hasattr(e, "children"):
            for c in e.children:
                visit(c)
            nd = OraNode()
            nd.kind = 1 if type(e).__name__ == "And" else 2     # ORA_NODE_AND / ORA_NODE_OR
            nd.n_children = len(e.children)
            nodes.append(nd)
            return
        nd = OraNode()
        nd.kind, nd.op, nd.col = 0, int(e.op), int(e.col)
        nd.param_begin, nd.n_params, nd.n_children = len(params), len(e.params), 0
        for v in e.params:
            p = OraParam()
            if v is None:
                p.is_null = 1
            elif isinstance(v, (bytes, bytearray)):
                b = bytes(v)
                keep.append(b)
                p.ptr, p.len = b, len(b)
            else:
                iv = int(v)
                p.i64 = iv - (1 << 64) if iv >= 1 << 63 else iv
            params.append(p)
        nodes.append(nd)

    visit(expr)
    node_arr = (OraNode * len(nodes))(*nodes)
    param_arr = (OraParam * max(len(params), 1))(*params)
    f = OraFilter()
    f.nodes, f.n_nodes = node_arr, len(nodes)
    f.params, f.n_params = param_arr, len(params)
    return f, (node_arr, param_arr, keep)


def cs_transform(buf: np.ndarray) -> np.ndarray:
    """CS block -> the same block with every integer stream restated as RAW (ora_cs_transform)."""
    L = oracle()
    L.ora_cs_transform.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
    src = np.ascontiguousarray(buf, dtype=np.uint8)
    n = C.c_int64(0)
    ora_check(L.ora_cs_transform(src.ctypes.data, src.size, None, 0, C.byref(n)), "ora_cs_transform(size)")
    out = np.zeros(n.value, dtype=np.uint8)
    ora_check(L.ora_cs_transform(src.ctypes.data, src.size, out.ctypes.data, out.size, C.byref(n)), "ora_cs_transform")
    return out[:n.value]


def cs_transform_table(table):
    """Every block of a CS table through cs_transform: a new TableImage (128-byte aligned blocks)."""
    from oceanbase_b200.sstable import TableImage
    parts, offs, sizes, pos = [], [], [], 0
    for i in range(table.n_blocks):
        t = cs_transform(table.block(i))
        pad = (-len(t)) % 128
        offs.append(pos)
        sizes.append(len(t))
        parts.append(t)
        if pad:
            parts.append(np.zeros(pad, dtype=np.uint8))
        pos += len(t) + pad
    return TableImage(np.concatenate(parts), np.array(offs, dtype=np.int64), np.array(sizes, dtype=np.int64), table.total_rows,
                      table.n_cols)


class Block:
    """One parsed micro-block view for the oracle."""

    def __init__(self, buf: np.ndarray):
        self.buf = np.ascontiguousarray(buf, dtype=np.uint8)
        self.b = OraBlock()
        ora_check(oracle().ora_block_init(C.byref(self.b), self.buf.ctypes.data, self.buf.size), "ora_block_init")
        self.row_count = self.b.row_count
        self.column_count = self.b.column_count

    def verify_checksums(self):
        return oracle().ora_block_verify_checksums(C.byref(self.b))

    def cell(self, col, row):
        d = OraDatum()
        ora_check(oracle().ora_decode_cell(C.byref(self.b), col, row, C.byref(d)), "ora_decode_cell")
        if d.is_null:
            return None
        if d.ptr:
            off = d.ptr - self.buf.ctypes.data
            if off < 0 or off + d.len > self.buf.size:   # a string a codec rebuilt: it lives in the oracle's arena
                return C.string_at(d.ptr, d.len)
            return bytes(self.buf[off:off + d.len])
        if d.len and d.ival == 0 and False:
            return 0
        return d.ival if d.len else b""

    # dictionary surface
    def dict_count(self, col):
        n = C.c_int64(0)
        ora_check(oracle().ora_dict_count(C.byref(self.b), col, C.byref(n)), "ora_dict_count")
        return n.value

    def dict_entry(self, col, ref):
        """bytes for strings, int (64-bit image) for integer classes"""
        d = OraDatum()
        ora_check(oracle().ora_dict_entry(C.byref(self.b), col, ref, C.byref(d)), "ora_dict_entry")
        if d.ptr:
            off = d.ptr - self.buf.ctypes.data
            return bytes(self.buf[off:off + d.len]), off
        return (d.ival if d.len else b""), None

    def dict_refs(self, col, row_ids):
        rid = np.ascontiguousarray(row_ids, dtype=np.int32)
        refs = np.zeros(max(len(rid), 1), dtype=np.uint32)
        ora_check(oracle().ora_dict_refs(C.byref(self.b), col, rid.ctypes.data, len(rid), refs.ctypes.data), "ora_dict_refs")
        return refs[:len(rid)]

    def cell_raw(self, col, row):
        d = OraDatum()
        ora_check(oracle().ora_decode_cell(C.byref(self.b), col, row, C.byref(d)), "ora_decode_cell")
        return d

    def get_rows_fixed(self, col, row_ids, elem_len=8, vec_offset=0, data=None, nulls=None):
        rid = np.ascontiguousarray(row_ids, dtype=np.int32)
        total = vec_offset + len(rid)
        if data is None:
            data = np.zeros(total * elem_len, dtype=np.uint8)
        if nulls is None:
            nulls = np.zeros((total + 63) // 64, dtype=np.uint64)
        hn = C.c_int32(0)
        ora_check(oracle().ora_get_rows_fixed(C.byref(self.b), col, rid.ctypes.data, len(rid), vec_offset,
                                              data.ctypes.data, elem_len, nulls.ctypes.data, C.byref(hn)),
                  "ora_get_rows_fixed")
        return data, nulls, hn.value

    def get_rows_discrete(self, col, row_ids, vec_offset=0, absolute=False):
        rid = np.ascontiguousarray(row_ids, dtype=np.int32)
        total = vec_offset + len(rid)
        ptrs = np.zeros(total, dtype=np.uint64)
        lens = np.zeros(total, dtype=np.int32)
        nulls = np.zeros((total + 63) // 64, dtype=np.uint64)
        hn = C.c_int32(0)
        ora_check(oracle().ora_get_rows_discrete(C.byref(self.b), col, rid.ctypes.data, len(rid), vec_offset,
                                                 ptrs.ctypes.data, lens.ctypes.data, nulls.ctypes.data, C.byref(hn)),
                  "ora_get_rows_discrete")
        if absolute:   # strings a codec rebuilt live in the oracle's arena: no block offset exists for them
            return ptrs, lens, nulls, hn.value
        # pointers -> offsets inside the block buffer
        offs = np.where(ptrs != 0, ptrs - np.uint64(self.buf.ctypes.data), 0).astype(np.uint64)
        return offs, lens, nulls, hn.value

    def filter_tree(self, expr, start=0, count=None):
        f, keep = ora_flatten_filter(expr)
        if count is None:
            count = self.row_count - start
        out = np.zeros(max(count, 1), dtype=np.uint8)
        ora_check(oracle().ora_filter_tree(C.byref(self.b), C.byref(f), start, count, out.ctypes.data),
                  "ora_filter_tree")
        return out[:count]


def bitmap_get_row_ids(bitmap, start, to, limit, id_offset=0):
    bm = np.ascontiguousarray(bitmap, dtype=np.uint8)
    out = np.zeros(max(limit, 1), dtype=np.int32)
    frm, cnt = C.c_int64(start), C.c_int64(0)
    code = oracle().ora_bitmap_get_row_ids(bm.ctypes.data, bm.size, out.ctypes.data, C.byref(cnt), C.byref(frm), to,
                                           limit, id_offset)
    ora_check(code, "ora_bitmap_get_row_ids")
    return out[:cnt.value].copy(), frm.value


def scan_table(table, filter_expr, proj_cols, proj_is_string, proj_elem_len, batch_size=256, want_row_ids=True,
               string_base=0):
    """Full-path oracle scan of a TableImage. Returns dict with dense outputs."""
    L = oracle()
    f, keep = ora_flatten_filter(filter_expr)
    n_proj = len(proj_cols)
    cap = table.total_rows
    datas, lens, nulls = [], [], []
    for i in range(n_proj):
        if proj_is_string[i]:
            datas.append(np.zeros(max(cap, 1), dtype=np.uint64))
            lens.append(np.zeros(max(cap, 1), dtype=np.int32))
        else:
            dt = {8: np.uint64, 4: np.uint32, 1: np.uint8}[proj_elem_len[i]]
            datas.append(np.zeros(max(cap, 1), dtype=dt))
            lens.append(None)
        nulls.append(np.zeros(max((cap + 63) // 64, 1), dtype=np.uint64))
    has_null = np.zeros(max(n_proj, 1), dtype=np.int32)
    row_ids = np.zeros(max(cap, 1), dtype=np.int32)
    sel_off = np.zeros(table.n_blocks + 1, dtype=np.int64)
    out = OraScanOut()
    da = (C.c_void_p * max(n_proj, 1))(*[d.ctypes.data for d in datas])
    la = (C.c_void_p * max(n_proj, 1))(*[(l.ctypes.data if l is not None else None) for l in lens])
    na = (C.c_void_p * max(n_proj, 1))(*[n.ctypes.data for n in nulls])
    out.data, out.lens, out.nulls = da, la, na
    out.has_null = has_null.ctypes.data
    out.row_ids = row_ids.ctypes.data if want_row_ids else None
    out.sel_offset = sel_off.ctypes.data
    out.cap_rows = cap
    out.string_base = string_base
    proj = np.ascontiguousarray(proj_cols, dtype=np.int32)
    total, sel = C.c_int64(0), C.c_int64(0)
    offs = np.ascontiguousarray(table.offsets, dtype=np.int64)
    sizes = np.ascontiguousarray(table.sizes, dtype=np.int64)
    code = L.ora_scan_blocks(table.image.ctypes.data, offs.ctypes.data, sizes.ctypes.data, 0, table.n_blocks,
                             C.byref(f) if f is not None else None, proj.ctypes.data, n_proj, batch_size, 0,
                             C.byref(out), C.byref(total), C.byref(sel))
    ora_check(code, "ora_scan_blocks")
    n = sel.value
    return {"total_rows": total.value, "selected": n, "data": [d[:n] for d in datas],
            "lens": [(l[:n] if l is not None else None) for l in lens],
            "nulls": [x[:(n + 63) // 64] for x in nulls], "has_null": has_null[:n_proj].copy(),
            "row_ids": row_ids[:n], "sel_offset": sel_off}


def scan_strings(table, res, p, string_base=0):
    """Bytes of string column p of a scan_table() result (None for NULL rows): cells inside the image through string_base,
    strings a codec rebuilt (HEX / STRING_DIFF / STRING_PREFIX) through their absolute address in the oracle's arena."""
    out = []
    ptrs, lens, nulls = res["data"][p], res["lens"][p], res["nulls"][p]
    for i in range(res["selected"]):
        if (int(nulls[i // 64]) >> (i % 64)) & 1:
            out.append(None)
            continue
        a, n = int(ptrs[i]), int(lens[i])
        off = a - string_base
        if 0 <= off and off + n <= table.image.size:
            out.append(bytes(table.image[off:off + n]))
        else:
            out.append(C.string_at(a, n))
    return out


def arena_reset():
    oracle().ora_arena_reset()


def scan_table_mt(table, filter_expr, proj_cols, batch_size=256, n_threads=1, block_limit=None):
    L = oracle()
    f, keep = ora_flatten_filter(filter_expr)
    proj = np.ascontiguousarray(proj_cols, dtype=np.int32)
    offs = np.ascontiguousarray(table.offsets, dtype=np.int64)
    sizes = np.ascontiguousarray(table.sizes, dtype=np.int64)
    nb = table.n_blocks if block_limit is None else min(block_limit, table.n_blocks)
    total, sel, cs = C.c_int64(0), C.c_int64(0), C.c_uint64(0)
    code = L.ora_scan_blocks_mt(table.image.ctypes.data, offs.ctypes.data, sizes.ctypes.data, nb,
                                C.byref(f) if f is not None else None, proj.ctypes.data, len(proj_cols), batch_size,
                                n_threads, C.byref(total), C.byref(sel), C.byref(cs))
    ora_check(code, "ora_scan_blocks_mt")
    return total.value, sel.value, cs.value


# ---- major compaction merge -------------------------------------------------------------------------
def decode_column_ext(table, col):
    """(values int64, ext uint8) of every cell of integer column `col`, by the oracle's block decoder."""
    n = int(table.total_rows)
    vals = np.zeros(n, dtype=np.int64)
    ext = np.zeros(n, dtype=np.uint8)
    offs = np.ascontiguousarray(table.offsets, dtype=np.int64)
    sizes = np.ascontiguousarray(table.sizes, dtype=np.int64)
    rows = C.c_int64(0)
    ora_check(oracle().ora_decode_column_ext(table.image.ctypes.data, offs.ctypes.data, sizes.ctypes.data, len(offs), col,
                                             vals.ctypes.data, ext.ctypes.data, n, C.byref(rows)), "ora_decode_column_ext")
    assert rows.value == n
    return vals, ext


def major_merge(runs, n_cols, default_vals=None, default_null=None):
    """runs: list (oldest -> newest) of dicts {key, flag (or None), vals [n_cols], ext [n_cols]} of numpy
    arrays. Returns dict(key, vals, null, dropped, fused)."""
    arr = (OraMergeRun * len(runs))()
    keep = []
    total = 0
    for i, r in enumerate(runs):
        key = np.ascontiguousarray(r["key"], dtype=np.int64)
        flag = None if r.get("flag") is None else np.ascontiguousarray(r["flag"], dtype=np.uint8)
        vals = [np.ascontiguousarray(v, dtype=np.int64) for v in r["vals"]]
        ext = [np.ascontiguousarray(e, dtype=np.uint8) for e in r["ext"]]
        vp = (C.c_void_p * max(n_cols, 1))(*[v.ctypes.data for v in vals])
        ep = (C.c_void_p * max(n_cols, 1))(*[e.ctypes.data for e in ext])
        keep += [key, flag, vals, ext, vp, ep]
        arr[i].n = len(key)
        arr[i].key = key.ctypes.data
        arr[i].flag = flag.ctypes.data if flag is not None else None
        arr[i].vals = vp
        arr[i].ext = ep
        more = [np.ascontiguousarray(k, dtype=np.int64) for k in (r.get("more_keys") or [])]
        if more:
            mp = (C.c_void_p * len(more))(*[k.ctypes.data for k in more])
            keep += [more, mp]
            arr[i].more_keys = mp
            arr[i].n_more_keys = len(more)
        total += len(key)
    out_key = np.zeros(max(total, 1), dtype=np.int64)
    out_vals = [np.zeros(max(total, 1), dtype=np.int64) for _ in range(n_cols)]
    out_null = [np.zeros(max(total, 1), dtype=np.uint8) for _ in range(n_cols)]
    ovp = (C.c_void_p * max(n_cols, 1))(*[v.ctypes.data for v in out_vals])
    onp = (C.c_void_p * max(n_cols, 1))(*[v.ctypes.data for v in out_null])
    dv = None if default_vals is None else np.ascontiguousarray(default_vals, dtype=np.int64)
    dn = None if default_null is None else np.ascontiguousarray(default_null, dtype=np.uint8)
    rows = C.c_int64(0)
    stats = (C.c_int64 * 2)()
    n_more = len(runs[0].get("more_keys") or [])
    out_more = [np.zeros(max(total, 1), dtype=np.int64) for _ in range(n_more)]
    omp = (C.c_void_p * max(n_more, 1))(*[v.ctypes.data for v in out_more])
    ora_check(oracle().ora_major_merge_keys(arr, len(runs), n_cols, dv.ctypes.data if dv is not None else None,
                                            dn.ctypes.data if dn is not None else None, total, out_key.ctypes.data, omp, ovp, onp,
                                            C.byref(rows), stats), "ora_major_merge_keys")
    n = rows.value
    return {"key": out_key[:n], "more_keys": [v[:n] for v in out_more], "vals": [v[:n] for v in out_vals],
            "null": [v[:n] for v in out_null], "dropped": stats[0], "fused": stats[1]}


# ---- skip index -------------------------------------------------------------------------------------------
def agg_row_read(row, col_idx, col_type):
    """ObAggRowReader::read: (bytes or None, is_prefix)."""
    buf = np.ascontiguousarray(row, dtype=np.uint8)
    ptr, ln, pre = C.c_void_p(), C.c_int32(0), C.c_int32(0)
    ora_check(oracle().ora_agg_row_read(buf.ctypes.data, buf.size, col_idx, col_type, C.byref(ptr), C.byref(ln),
                                        C.byref(pre)), "ora_agg_row_read")
    if not ptr.value:
        return None, False
    off = ptr.value - buf.ctypes.data
    return bytes(buf[off:off + ln.value]), bool(pre.value)


def skip_index_filter(row, row_count, col_types, expr):
    """ObSSTableIndexFilter::check_range on one block's aggregate row: ORA_MASK_* (0 uncertain, 1 true, 2 false)."""
    f, keep = ora_flatten_filter(expr)
    buf = np.ascontiguousarray(row, dtype=np.uint8) if row is not None and len(row) else None
    types = np.ascontiguousarray(col_types, dtype=np.uint8)
    mask = C.c_int32(0)
    ora_check(oracle().ora_skip_index_filter(buf.ctypes.data if buf is not None else None, buf.size if buf is not None else 0,
                                             row_count, types.ctypes.data, len(types), C.byref(f), C.byref(mask)),
              "ora_skip_index_filter")
    return mask.value
