"""ctypes binding of libobgpu_scan.so (include/obgpu_scan.h). Fails loudly when the library is
missing: the product has no CPU path."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
lib_path = os.path.join(_HERE, "csrc", "libobgpu_scan.so")
writer_lib_path = os.path.join(_HERE, "csrc", "libobgpu_writer.so")

OB_SUCCESS = 0
OB_INVALID_ARGUMENT = -4002
OB_NOT_SUPPORTED = -4007
OB_ERR_SYS = -4015
OB_BUF_NOT_ENOUGH = -4024
OB_INVALID_DATA = -4070

(WHITE_OP_EQ, WHITE_OP_LE, WHITE_OP_LT, WHITE_OP_GE, WHITE_OP_GT, WHITE_OP_NE, WHITE_OP_BT,
 WHITE_OP_IN, WHITE_OP_NU, WHITE_OP_NN) = range(10)
ENC_RAW, ENC_DICT, ENC_RLE, ENC_CONST, ENC_INTEGER_BASE_DIFF, ENC_STRING_DIFF, ENC_HEX_PACKING, ENC_STRING_PREFIX, ENC_COLUMN_EQUAL, ENC_COLUMN_SUBSTR = range(10)
ENC_CS_INTEGER, ENC_CS_INT_DICT, ENC_CS_STRING, ENC_CS_STR_DICT = 16, 17, 18, 19  # columns of a CS_ENCODING_ROW_STORE block
ENC_CS_AUTO = 33  # writer only, CS blocks: INTEGER vs INT_DICT / STRING vs STR_DICT (ObMicroBlockCSEncoder::choose_encoder_)
ENC_AUTO = 32  # writer only: codec chosen per micro-block (ObMicroBlockEncoder::choose_encoder)
OBJ_TINYINT, OBJ_SMALLINT, OBJ_MEDIUMINT, OBJ_INT32, OBJ_INT = 1, 2, 3, 4, 5
OBJ_UTINYINT, OBJ_USMALLINT, OBJ_UMEDIUMINT, OBJ_UINT32, OBJ_UINT64 = 6, 7, 8, 9, 10
OBJ_DATETIME, OBJ_TIMESTAMP, OBJ_DATE, OBJ_TIME, OBJ_YEAR, OBJ_VARCHAR, OBJ_CHAR = 17, 18, 19, 20, 21, 22, 23
NODE_WHITE, NODE_AND, NODE_OR = 0, 1, 2


def datum_len_of(obj_type: int) -> int:
    """Datum length of an integer-class ObObjType (ObDatum::get_obj_datum_map_type): year 1, date 4, else 8."""
    return 1 if obj_type == OBJ_YEAR else (4 if obj_type == OBJ_DATE else 8)


class ObGpuError(RuntimeError):
    def __init__(self, code, what, detail=""):
        self.code = code
        super().__init__(f"{what} failed: OB error {code}" + (f" ({detail})" if detail else ""))


class FilterParam(C.Structure):
    _fields_ = [("i64", C.c_int64), ("ptr", C.c_char_p), ("len", C.c_uint32), ("is_null", C.c_int32)]


class FilterNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("op", C.c_int32), ("col", C.c_int32), ("param_begin", C.c_int32),
                ("n_params", C.c_int32), ("n_children", C.c_int32)]


class Filter(C.Structure):
    _fields_ = [("nodes", C.POINTER(FilterNode)), ("n_nodes", C.c_int32),
                ("params", C.POINTER(FilterParam)), ("n_params", C.c_int32)]


class ScanSpec(C.Structure):
    _fields_ = [("filter", C.POINTER(Filter)), ("proj_cols", C.POINTER(C.c_int32)), ("n_proj", C.c_int32),
                ("want_row_ids", C.c_int32), ("string_base", C.c_uint64), ("max_selected_rows", C.c_int64)]


class ResultInfo(C.Structure):
    _fields_ = [("total_rows", C.c_int64), ("selected_rows", C.c_int64), ("n_blocks", C.c_int32),
                ("n_proj", C.c_int32)]


class ResultCol(C.Structure):
    _fields_ = [("data", C.c_void_p), ("aux", C.c_void_p), ("nulls", C.c_void_p), ("elem_len", C.c_int32),
                ("is_string", C.c_int32), ("has_null", C.c_int32), ("obj_type", C.c_int32)]


class HostAgg(C.Structure):
    _fields_ = [("kind", C.c_int32), ("col_a", C.c_int32), ("col_b", C.c_int32)]


class HostScanSpec(C.Structure):
    _fields_ = [("image", C.c_void_p), ("image_size", C.c_int64), ("offsets", C.c_void_p), ("sizes", C.c_void_p),
                ("n_blocks", C.c_int32), ("filter", C.POINTER(Filter)), ("proj_cols", C.POINTER(C.c_int32)), ("n_proj", C.c_int32),
                ("blocks_per_batch", C.c_int32), ("ramp", C.c_int32), ("selectivity_hint", C.c_double), ("string_base", C.c_uint64),
                ("agg_rows", C.c_void_p), ("agg_off", C.c_void_p), ("out_data", C.POINTER(C.c_void_p)),
                ("out_lens", C.POINTER(C.c_void_p)), ("out_nulls", C.POINTER(C.c_void_p)), ("out_cap_rows", C.c_int64),
                ("out_row_ids", C.c_void_p), ("out_block_begin", C.c_void_p), ("out_block_count", C.c_void_p),
                ("no_row_output", C.c_int32), ("aggs", C.POINTER(HostAgg)), ("n_aggs", C.c_int32), ("zero_copy", C.c_int32)]


class HostScanResult(C.Structure):
    _fields_ = [("total_rows", C.c_int64), ("selected_rows", C.c_int64), ("n_batches", C.c_int32),
                ("batch_row_begin", C.c_void_p), ("batch_rows", C.c_void_p), ("batch_block_begin", C.c_void_p),
                ("n_batches_cap", C.c_int32), ("agg_out", (C.c_int64 * 2) * 16), ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64), ("kernel_launches", C.c_int64)]


class StreamRun(C.Structure):
    _fields_ = [("image", C.c_void_p), ("offsets", C.c_void_p), ("sizes", C.c_void_p), ("end_keys", C.c_void_p), ("n_blocks", C.c_int32)]


MERGE_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int32, C.c_void_p)


class ColInput(C.Structure):
    _fields_ = [("obj_type", C.c_int32), ("encoding", C.c_int32), ("i64", C.c_void_p), ("is_null", C.c_void_p),
                ("str_heap", C.c_void_p), ("str_off", C.c_void_p), ("byte_packing_only", C.c_int32),
                ("ref_col", C.c_int32)]


class AggCell(C.Structure):
    _fields_ = [("col_idx", C.c_uint32), ("col_type", C.c_uint8), ("is_null", C.c_uint8), ("is_prefix", C.c_uint8),
                ("reserved", C.c_uint8), ("len", C.c_int32), ("data", C.c_void_p)]


SK_IDX_MIN, SK_IDX_MAX, SK_IDX_NULL_COUNT, SK_IDX_SUM = range(4)           # blocksstable::ObSkipIndexColType
BOOL_MASK_UNCERTAIN, BOOL_MASK_ALWAYS_TRUE, BOOL_MASK_ALWAYS_FALSE = range(3)  # sql::ObBoolMaskType
AGG_COUNT, AGG_SUM, AGG_SUM_PRODUCT, AGG_MIN, AGG_MAX = range(5)
DF_NOT_EXIST, DF_LOCK, DF_UPDATE, DF_INSERT, DF_DELETE = range(5)  # blocksstable::ObDmlFlag


class MergeRun(C.Structure):
    _fields_ = [("n", C.c_int64), ("key", C.c_void_p), ("flag", C.c_void_p), ("vals", C.POINTER(C.c_void_p)),
                ("ext", C.POINTER(C.c_void_p)), ("more_keys", C.POINTER(C.c_void_p)), ("n_more_keys", C.c_int32)]


class MacroSpec(C.Structure):
    _fields_ = [("tablet_id", C.c_uint64), ("logical_version", C.c_int64), ("first_data_seq", C.c_int64), ("header_version", C.c_int32),
                ("is_cg", C.c_int32), ("rowkey_col_cnt", C.c_int32), ("n_cols", C.c_int32), ("col_metas", C.c_void_p),
                ("col_orders", C.c_void_p), ("macro_block_size", C.c_int64)]


class EncodeCol(C.Structure):
    _fields_ = [("dev_vals", C.c_void_p), ("dev_null", C.c_void_p), ("obj_type", C.c_int32), ("byte_packing_only", C.c_int32)]


class EncodedInfo(C.Structure):
    _fields_ = [("image_size", C.c_int64), ("total_rows", C.c_int64), ("n_blocks", C.c_int32), ("n_host_blocks", C.c_int32)]


class MergeInfo(C.Structure):
    _fields_ = [("in_rows", C.c_int64), ("out_rows", C.c_int64), ("dropped_deletes", C.c_int64),
                ("fused_rows", C.c_int64)]


def writer_signatures():
    """name -> (restype, argtypes) for every symbol include/obgpu_writer.h declares (libobgpu_writer.so)."""
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    P = C.POINTER
    return {
        "obgpu_writer_block_bound": (i64, [P(ColInput), i32, i64, i64]),
        "obgpu_writer_encode_block": (C.c_int, [P(ColInput), i32, i32, i64, i64, vp, i64, P(i64)]),
        "obgpu_writer_encode_table": (C.c_int, [P(ColInput), i32, i32, i64, i64, i32, i32, P(vp)]),
        "obgpu_table_image_info": (C.c_int, [vp, P(i64), P(i32)]),
        "obgpu_table_image_export": (C.c_int, [vp, vp, i64, vp, vp, i32]),
        "obgpu_table_image_free": (None, [vp]),
        "obgpu_agg_row_write": (C.c_int, [P(AggCell), i32, i32, vp, i64, P(i64)]),
        "obgpu_writer_block_agg_row": (C.c_int, [P(ColInput), i32, vp, i32, i64, i64, vp, i64, P(i64)]),
        "obgpu_writer_table_agg_rows": (C.c_int, [P(ColInput), i32, vp, i32, i64, i64, vp, i64, vp, P(i64)]),
        "obgpu_writer_set_cs_stream_encoding": (C.c_int, [i32]),
        "obgpu_writer_build_macro_blocks": (C.c_int, [vp, vp, vp, i32, P(MacroSpec), vp, i64, P(i64), P(i32), vp, i32]),
        "obgpu_writer_stream_encode": (C.c_int, [i32, i32, vp, i64, vp, i64, P(i64)]),
    }


def declared_signatures():
    """name -> (restype, argtypes) for every symbol include/obgpu_scan.h, include/obgpu_compaction.h and
    include/obgpu_skip_index.h declare (libobgpu_scan.so)."""
    vp, i32, i64, u64 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64
    P = C.POINTER
    return {
        "obgpu_ctx_create": (C.c_int, [C.c_int, P(vp)]),
        "obgpu_ctx_destroy": (None, [vp]),
        "obgpu_ctx_set_stream": (C.c_int, [vp, vp]),
        "obgpu_ctx_synchronize": (C.c_int, [vp]),
        "obgpu_ctx_last_error": (C.c_char_p, [vp]),
        "obgpu_ctx_launch_count": (i64, [vp]),
        "obgpu_ctx_set_profiling": (C.c_int, [vp, i32]),
        "obgpu_ctx_kernel_times": (C.c_int, [vp, vp, i32, P(i32)]),
        "obgpu_comm_unique_id": (C.c_int, [vp]),
        "obgpu_comm_create": (C.c_int, [vp, vp, i32, i32, P(vp)]),
        "obgpu_comm_destroy": (None, [vp]),
        "obgpu_merge_decoded_distributed": (C.c_int, [vp, vp, P(MergeRun), vp, i32, i32, i32, i32, vp, vp, i32, P(vp), vp, vp]),
        "obgpu_pipeline_create": (C.c_int, [C.c_int, i32, P(vp)]),
        "obgpu_pipeline_destroy": (None, [vp]),
        "obgpu_pipeline_last_error": (C.c_char_p, [vp]),
        "obgpu_pipeline_plan": (C.c_int, [P(HostScanSpec), P(i32), P(i64)]),
        "obgpu_pipeline_scan": (C.c_int, [vp, P(HostScanSpec), P(HostScanResult)]),
        "obgpu_batch_open": (C.c_int, [vp, vp, i64, vp, vp, i32, i32, vp, P(vp)]),
        "obgpu_batch_close": (None, [vp]),
        "obgpu_batch_block_info": (C.c_int, [vp, i32, P(i64), P(i32)]),
        "obgpu_batch_total_rows": (C.c_int, [vp, P(i64)]),
        "obgpu_scan": (C.c_int, [vp, P(ScanSpec), P(vp)]),
        "obgpu_result_free": (None, [vp]),
        "obgpu_result_info_get": (C.c_int, [vp, P(ResultInfo)]),
        "obgpu_result_col_get": (C.c_int, [vp, i32, P(ResultCol)]),
        "obgpu_result_block_tables": (C.c_int, [vp, P(vp), P(vp), P(vp), P(vp)]),
        "obgpu_result_fetch_col": (C.c_int, [vp, i32, i64, i64, vp, vp, vp]),
        "obgpu_result_fetch_cols": (C.c_int, [vp, i32, vp, i64, i64, vp, vp, vp]),
        "obgpu_result_aggregate": (C.c_int, [vp, i32, i32, i32, vp]),
        "obgpu_result_fetch_sel_offsets": (C.c_int, [vp, vp]),
        "obgpu_result_fetch_row_ids": (C.c_int, [vp, i64, i64, vp]),
        "obgpu_result_fetch_bitmap": (C.c_int, [vp, i32, i64, i64, vp]),
        "obgpu_filter_white": (C.c_int, [vp, i32, i32, i32, P(FilterParam), i32, i64, i64, vp]),
        "obgpu_filter_tree": (C.c_int, [vp, i32, P(Filter), i64, i64, vp]),
        "obgpu_bitmap_to_row_ids": (C.c_int, [vp, vp, i64, P(i64), i64, i64, i64, vp, P(i64)]),
        "obgpu_project_fixed": (C.c_int, [vp, i32, i32, vp, i64, i64, vp, i32, vp, P(i32)]),
        "obgpu_project_discrete": (C.c_int, [vp, i32, i32, vp, i64, i64, u64, vp, vp, vp, P(i32)]),
        "obgpu_project_datums": (C.c_int, [vp, i32, i32, vp, i64, i64, u64, vp]),
        "obgpu_result_fetch_datums": (C.c_int, [vp, i32, i64, i64, vp, vp]),
        "obgpu_cg_bitmap_create": (C.c_int, [vp, i64, i32, P(vp)]),
        "obgpu_cg_bitmap_free": (None, [vp]),
        "obgpu_cg_bitmap_apply_result": (C.c_int, [vp, vp, i64, i32]),
        "obgpu_cg_bitmap_popcnt": (C.c_int, [vp, i64, i64, P(i64)]),
        "obgpu_cg_bitmap_fetch": (C.c_int, [vp, i64, i64, vp]),
        "obgpu_scan_bitmap": (C.c_int, [vp, vp, i64, vp, P(vp)]),
        "obgpu_batch_column_materialised": (C.c_int, [vp, i32, P(i32)]),
        "obgpu_result_fetch_strings": (C.c_int, [vp, i32, i64, i64, vp, i64, vp, P(i64)]),
        "obgpu_project_strings": (C.c_int, [vp, i32, i32, vp, i64, vp, i64, vp, vp, P(i32), P(i64)]),
        "obgpu_batch_column_type": (C.c_int, [vp, i32, P(i32), P(i32)]),
        "obgpu_block_distinct_count": (C.c_int, [vp, i32, i32, P(i64)]),
        "obgpu_block_read_distinct": (C.c_int, [vp, i32, i32, u64, vp, vp, i64, P(i64)]),
        "obgpu_block_read_reference": (C.c_int, [vp, i32, i32, vp, i64, vp]),
        "obgpu_filter_dict_pass": (C.c_int, [vp, i32, i32, vp, i64, i32, i64, i64, vp]),
        "obgpu_block_group_by": (C.c_int, [vp, i32, i32, vp, i32, vp, i64, vp, i64, P(i64)]),
        "obgpu_result_group_by": (C.c_int, [vp, i32, vp, i32, vp, vp, i64, P(i64)]),
        "obgpu_version": (C.c_char_p, []),
        # include/obgpu_compaction.h
        "obgpu_batch_decode_column": (C.c_int, [vp, i32, vp, vp]),
        "obgpu_batch_decode_columns": (C.c_int, [vp, i32, vp, vp, vp]),
        "obgpu_batch_decode_columns_tagged": (C.c_int, [vp, i32, vp, i32, vp, vp]),
        "obgpu_merge_result_set_string_images": (C.c_int, [vp, vp, vp, i32]),
        "obgpu_merge_runs_streamed": (C.c_int, [i32, i32, vp, i32, i32, i32, vp, i32, vp, vp, i32, MERGE_SINK, vp, P(i32)]),
        "obgpu_merge_result_fetch_strings": (C.c_int, [vp, i32, i64, i64, vp, i64, vp, vp, P(i64)]),
        "obgpu_merge_decoded": (C.c_int, [vp, P(MergeRun), i32, i32, vp, vp, P(vp)]),
        "obgpu_merge_runs": (C.c_int, [vp, P(vp), i32, i32, i32, vp, i32, vp, vp, P(vp)]),
        "obgpu_merge_runs_keys": (C.c_int, [vp, P(vp), i32, vp, i32, i32, vp, i32, vp, vp, P(vp)]),
        "obgpu_merge_result_free": (None, [vp]),
        "obgpu_merge_result_info": (C.c_int, [vp, P(MergeInfo)]),
        "obgpu_merge_result_cols": (C.c_int, [vp, P(vp), P(P(vp)), P(P(vp))]),
        "obgpu_merge_result_fetch": (C.c_int, [vp, i32, i64, i64, vp, vp]),
        "obgpu_batch_open_macro_blocks": (C.c_int, [vp, vp, i64, i64, i32, i32, P(vp), P(i32)]),
        "obgpu_encode_columns": (C.c_int, [vp, P(EncodeCol), i32, i32, i64, i64, i32, P(vp)]),
        "obgpu_merge_result_encode": (C.c_int, [vp, vp, vp, i32, i32, i64, i32, P(vp)]),
        "obgpu_encode_columns_with": (C.c_int, [vp, P(EncodeCol), vp, i32, i32, i64, i64, i32, P(vp)]),
        "obgpu_merge_result_encode_with": (C.c_int, [vp, vp, vp, vp, i32, i32, i64, i32, P(vp)]),
        "obgpu_encoded_get_info": (C.c_int, [vp, P(EncodedInfo)]),
        "obgpu_encoded_fetch": (C.c_int, [vp, vp, i64, vp, vp, i32]),
        "obgpu_encoded_device_image": (C.c_int, [vp, P(vp), P(vp), P(vp)]),
        "obgpu_encoded_column_checksums": (C.c_int, [vp, vp]),
        "obgpu_encoded_free": (None, [vp]),
        "obgpu_column_checksums": (C.c_int, [vp, P(EncodeCol), i32, i64, vp]),
        # include/obgpu_skip_index.h
        "obgpu_batch_set_agg_rows": (C.c_int, [vp, vp, vp]),
        "obgpu_batch_skip_index_filter": (C.c_int, [vp, P(Filter), vp]),
        "obgpu_result_skip_info": (C.c_int, [vp, P(i64), P(i64)]),
    }


def _load(path, signatures):
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). oceanbase_b200 has no CPU fallback.")
    L = C.CDLL(path)
    for name, (res, args) in signatures.items():
        fn = getattr(L, name)  # AttributeError => the library does not export the declared ABI
        fn.restype = res
        fn.argtypes = args
    return L


class _Libs:
    """Symbol lookup over the two in-tree libraries: the writer entry points resolve to libobgpu_writer.so
    (plain C++), everything else to the CUDA product library, which is only mapped on first use."""

    def __init__(self):
        self.writer = _load(writer_lib_path, writer_signatures())
        self._scan = None
        self._wnames = set(writer_signatures())

    @property
    def scan(self):
        if self._scan is None:
            self._scan = _load(lib_path, declared_signatures())
        return self._scan

    def __getattr__(self, name):
        if name.startswith("obgpu_"):
            return getattr(self.writer if name in self._wnames else self.scan, name)
        raise AttributeError(name)


lib = _Libs()   # the first product call raises ImportError when libobgpu_scan.so is missing: no CPU path exists


def check(code, what, ctx=None):
    if code != OB_SUCCESS:
        detail = ""
        try:
            if ctx is not None:   # writer calls have no ctx (and must not map the CUDA library)
                detail = (lib.obgpu_ctx_last_error(ctx) or b"").decode()
        except Exception:  # pragma: no cover
            pass
        raise ObGpuError(code, what, detail)
