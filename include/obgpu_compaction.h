/* obgpu_compaction.h -- C-ABI of the B200-native major-compaction merge.
 *
 * Drop-in boundary for the reference's partition merger
 *   compaction/ob_partition_merger.cpp:678-829   ObPartitionMajorMerger::merge_partition
 *   compaction/ob_partition_rows_merger.cpp:815  ObPartitionMergeHelper::find_rowkey_minimum_iters
 *   compaction/ob_partition_merge_fuser.cpp:106  ObMergeFuser::fuse_row (+ :284 end_fuse_row)
 *   storage/ob_row_fuse.cpp:191-275              ObRowFuse::fuse_row (NOP fill, delete stops the fuse)
 *   compaction/ob_partition_merger.cpp:648-676   inner_process (delete rows are dropped in a major merge)
 * K sorted runs (one per table of the merge, table index ascending = older -> newer) are merged by
 * rowkey; rows with the same rowkey are fused newest first; the result is the ordered row stream the
 * reference hands to ObMacroBlockWriter::append_row. The runs arrive as decoded column arrays in HBM
 * (obgpu_batch_decode_column turns an opened page batch into them), so the same entry point serves a
 * single GPU and the range-partitioned multi-GPU merge (each rank merges the slices it received).
 *
 * Same conventions as obgpu_scan.h: int OB codes, no exceptions, caller-owned outputs. */
#ifndef OBGPU_COMPACTION_H_
#define OBGPU_COMPACTION_H_

#include "obgpu_scan.h"

#ifdef __cplusplus
extern "C" {
#endif

/* blocksstable::ObDmlFlag (storage/blocksstable/ob_datum_row.h) */
enum {
  OBGPU_DF_NOT_EXIST = 0,
  OBGPU_DF_LOCK = 1,
  OBGPU_DF_UPDATE = 2,
  OBGPU_DF_INSERT = 3,
  OBGPU_DF_DELETE = 4
};

#define OBGPU_MERGE_MAX_RUNS 64
#define OBGPU_MERGE_MAX_COLS 64
#define OBGPU_MERGE_MAX_KEY_COLS 8

/* All cells of column `col` (integer class, or string class as references -- see below) of an opened batch, in row order, into caller-owned DEVICE
 * buffers of total_rows entries: value image (what the reference would MEMCPY into the datum, 0 for
 * ext cells) and ext (0 value, 1 NULL, 2 NOP -- ObStoredExtValue). Runs on the ctx stream. */
int obgpu_batch_decode_column(obgpu_batch *batch, int32_t col, int64_t *dev_vals, uint8_t *dev_ext);
/* Up to 16 columns with one launch and one synchronisation (each block image is read once). */
int obgpu_batch_decode_columns(obgpu_batch *batch, int32_t n_cols, const int32_t *cols,
                               int64_t *const *dev_vals, uint8_t *const *dev_ext);

/* String-class columns: the "value image" of a cell is a REFERENCE into the run's page batch,
 *     ref = (tag << 58) | (byte offset of the cell inside the batch image << 22) | length
 * (tag < 64, offset < 2^36, length < 2^22; larger cells report OBGPU_NOT_SUPPORTED). The merge moves references like
 * integer cells; obgpu_merge_result_fetch_strings turns them back into bytes. `string_tag` names the run the batch
 * belongs to (obgpu_merge_runs uses the run index); obgpu_batch_decode_columns is the tag-0 form. */
int obgpu_batch_decode_columns_tagged(obgpu_batch *batch, int32_t n_cols, const int32_t *cols, int32_t string_tag,
                                      int64_t *const *dev_vals, uint8_t *const *dev_ext);

/* One sorted run, decoded, resident in HBM (all pointers are device pointers; the vals / ext
 * pointer ARRAYS themselves live in host memory). Rowkey: INT64 columns (`key`, plus
 * `more_keys` for a composite rowkey), ascending, unique inside the run. */
typedef struct obgpu_merge_run {
  int64_t n;
  const int64_t *key;
  const uint8_t *flag;         /* ObDmlFlag per row; NULL: every row DF_INSERT                  */
  const int64_t *const *vals;  /* [n_cols] value arrays                                           */
  const uint8_t *const *ext;   /* [n_cols] 0 value, 1 NULL, 2 NOP                                 */
  /* composite rowkeys: the rowkey columns after the first (INT64 images, no NULLs), compared column by column
   * after `key` like ObStorageDatumUtils does; the same count in every run, 0 for a single-column rowkey       */
  const int64_t *const *more_keys;
  int32_t n_more_keys;
} obgpu_merge_run;

typedef struct obgpu_merge_result obgpu_merge_result;

/* runs[0] is the oldest table, runs[n_runs - 1] the newest. default_vals / default_null: the
 * default row that fills cells still NOP after the fuse (ObMajorPartitionMergeFuser::end_fuse_row);
 * NULL pointers mean "every default is NULL". */
int obgpu_merge_decoded(obgpu_ctx *ctx, const obgpu_merge_run *runs, int32_t n_runs, int32_t n_cols,
                        const int64_t *default_vals, const uint8_t *default_null,
                        obgpu_merge_result **out);
void obgpu_merge_result_free(obgpu_merge_result *res);

/* The whole merge of one range from opened page batches (one per table, oldest first): decodes rowkey_col,
 * flag_col (-1: every row DF_INSERT) and the payload columns of every run into temporary device arrays and
 * calls obgpu_merge_decoded. This is the call the C++ adapter (oceanbase_b200/host/ob_gpu_partition_merger.h)
 * makes from ObPartitionMajorMerger::merge_partition. All batches must belong to `ctx`. */
int obgpu_merge_runs(obgpu_ctx *ctx, obgpu_batch *const *runs, int32_t n_runs, int32_t rowkey_col,
                     int32_t flag_col, const int32_t *cols, int32_t n_cols, const int64_t *default_vals,
                     const uint8_t *default_null, obgpu_merge_result **out);

/* Same with a composite rowkey: rowkey_cols[0 .. n_rowkey_cols) in comparison order (at most OBGPU_MERGE_MAX_KEY_COLS). */
int obgpu_merge_runs_keys(obgpu_ctx *ctx, obgpu_batch *const *runs, int32_t n_runs, const int32_t *rowkey_cols,
                          int32_t n_rowkey_cols, int32_t flag_col, const int32_t *cols, int32_t n_cols,
                          const int64_t *default_vals, const uint8_t *default_null, obgpu_merge_result **out);

typedef struct obgpu_merge_info {
  int64_t in_rows;          /* rows of all runs                                              */
  int64_t out_rows;         /* rows of the merged stream                                     */
  int64_t dropped_deletes;  /* rowkeys whose fused row is a delete                           */
  int64_t fused_rows;       /* output rows fused from more than one run                      */
} obgpu_merge_info;
/* Synchronises the ctx stream and reads back the totals. */
int obgpu_merge_result_info(obgpu_merge_result *res, obgpu_merge_info *info);
/* Device pointers of the merged stream (valid until obgpu_merge_result_free): rowkeys [out_rows],
 * and per column values [out_rows] + null bytes (1 => NULL) [out_rows]. */
int obgpu_merge_result_cols(obgpu_merge_result *res, const int64_t **key_dev,
                            const int64_t *const **vals_dev, const uint8_t *const **null_dev);
/* Device -> host copy of rows [row_begin, row_begin + row_count) of column `col` (-1: the first rowkey column,
 * -2, -3, ...: the following rowkey columns of a composite rowkey). */
int obgpu_merge_result_fetch(obgpu_merge_result *res, int32_t col, int64_t row_begin,
                             int64_t row_count, int64_t *host_vals, uint8_t *host_null);

/* String columns of the merged stream (what ObMacroBlockWriter::append_row receives as ObString datums): cells
 * [row_begin, row_begin + row_count) of column `col` are copied back to back into host_heap, row i occupying
 * [host_off[i], host_off[i + 1]) (row_count + 1 offsets; a NULL cell is empty and flagged in host_null). *heap_bytes
 * receives the bytes needed; OBGPU_BUF_NOT_ENOUGH when heap_cap is smaller (nothing copied). The page batches the
 * references point into must still be open: obgpu_merge_runs records their images itself; after obgpu_merge_decoded
 * the caller names them (index = string tag) with their sizes; a reference that does not lie inside its image reports
 * OBGPU_INVALID_DATA instead of being followed. */
int obgpu_merge_result_set_string_images(obgpu_merge_result *res, const void *const *dev_images, const int64_t *image_sizes,
                                         int32_t n_images);
int obgpu_merge_result_fetch_strings(obgpu_merge_result *res, int32_t col, int64_t row_begin, int64_t row_count,
                                     void *host_heap, int64_t heap_cap, int64_t *host_off, uint8_t *host_null,
                                     int64_t *heap_bytes);

/* =============================================================================================
 * Multi-GPU: the range-partitioned merge (one rowkey range per rank, ObParallelMergeCtx,
 * compaction/ob_partition_parallel_merge_ctx.cpp:187-424). The exchange of run slices between the ranks is the one
 * collective step of the whole path: sampled splitters through ncclAllGather, slices through grouped
 * ncclSend / ncclRecv over NVLink, all enqueued on the ctx stream by the library (NCCL is bound with dlopen).
 * ============================================================================================= */
#define OBGPU_COMM_ID_BYTES 128
typedef struct obgpu_comm obgpu_comm;
/* Rank 0 makes the communicator id (ncclGetUniqueId) and hands its 128 bytes to every rank through the caller's own
 * channel; then every rank calls obgpu_comm_create with the same id. One process per GPU. */
int obgpu_comm_unique_id(void *id_out);
int obgpu_comm_create(obgpu_ctx *ctx, const void *id, int32_t rank, int32_t world, obgpu_comm **out);
void obgpu_comm_destroy(obgpu_comm *comm);
/* Every run index in [0, n_runs_total) is held (decoded, in HBM) by exactly one rank: local_runs[q] is run
 * run_index[q]. Collective over the communicator: splitters from samples_per_run evenly spaced rowkeys of every run,
 * every rank receives the slices of its rowkey range and merges them (obgpu_merge_decoded); the concatenation of the
 * ranks' results in rank order is the merged stream. Integer payload columns (string references are only valid on the
 * device that decoded them). Composite rowkeys partition on the first rowkey column. The local runs' arrays must stay
 * alive until the ctx stream has been synchronised (e.g. obgpu_merge_result_info). splitters_out: world - 1 values,
 * recv_rows_out: rows of every run in this rank's range (both optional, host). */
int obgpu_merge_decoded_distributed(obgpu_ctx *ctx, obgpu_comm *comm, const obgpu_merge_run *local_runs,
                                    const int32_t *run_index, int32_t n_local, int32_t n_runs_total, int32_t n_cols,
                                    int32_t n_more_keys, const int64_t *default_vals, const uint8_t *default_null,
                                    int32_t samples_per_run, obgpu_merge_result **out, int64_t *splitters_out,
                                    int64_t *recv_rows_out);

/* ---- runs larger than device memory: the merge range by range, copies of the next range under the merge of this one ----------
 * One run = its SSTable in HOST memory (pinned for full copy overlap) + the last rowkey of every micro-block (what the index rows
 * hold). The rowkey space is cut into n_ranges ranges at quantiles of the block end keys (ObParallelMergeCtx cuts parallel-merge
 * ranges at block boundaries of the index tree the same way, compaction/ob_partition_parallel_merge_ctx.cpp:187-424); for every
 * range the blocks of each run that can hold its rowkeys are copied, decoded, cut to the range and merged, and sink(arg, range, result)
 * is called with ranges 0, 1, 2 ... in rowkey order (the result is only valid inside the call: fetch / encode the rows there).
 * n_streams ranges are in flight on their own streams; device memory holds n_streams ranges whatever the size of the runs.
 * Single INT64 rowkey column, integer payload columns. */
typedef struct obgpu_stream_run {
  const void *image;         /* host memory, blocks 16-byte aligned */
  const int64_t *offsets;    /* [n_blocks] */
  const int64_t *sizes;      /* [n_blocks] */
  const int64_t *end_keys;   /* [n_blocks] last rowkey of every micro-block, ascending */
  int32_t n_blocks;
} obgpu_stream_run;
typedef int (*obgpu_merge_sink)(void *arg, int32_t range, obgpu_merge_result *result);
int obgpu_merge_runs_streamed(int device, int32_t n_streams, const obgpu_stream_run *runs, int32_t n_runs, int32_t rowkey_col,
                              int32_t flag_col /* -1: every row DF_INSERT */, const int32_t *cols, int32_t n_cols,
                              const int64_t *default_vals, const uint8_t *default_null, int32_t n_ranges, obgpu_merge_sink sink,
                              void *sink_arg, int32_t *ranges_done);

/* =============================================================================================
 * Phase B of the compaction: the merged rows leave the device as SSTable bytes, not as rows.
 *   blocksstable/encoding/ob_micro_block_encoder.cpp:561-721   ObMicroBlockEncoder::build_block (PAX layout)
 *   blocksstable/encoding/ob_raw_encoder.cpp:95-155            ObRawEncoder::traverse (width: bit / byte packing, ext bits)
 *   blocksstable/encoding/ob_encoding_util.cpp:37-73           get_packing_size
 *   blocksstable/ob_micro_block_header.cpp:193-233             header checksum; payload checksum = ob_crc64_sse42 (crc32c)
 *   blocksstable/ob_micro_block_checksum_helper.cpp:127-257    cal_column_checksum: per column, the wrapping int64 sum
 *                                                              over the rows of ObDatum::checksum(0) (share/datum/ob_datum.h:849)
 *   column_store/ob_co_merge_writer.cpp:67-117                 ObWriteHelper::project / append: one merged stream replayed into
 *                                                              the writer of every column group
 * Integer-class columns (device arrays of 8-byte value images + optional NULL bytes, 1 => NULL), every column RAW
 * (ObRawEncoder): consecutive blocks of rows_per_block rows, block i at offsets[i] (aligned to `align`, a power of two
 * >= 16, padding zeroed) -- byte for byte what obgpu_writer_encode_table (include/obgpu_writer.h) produces for the same
 * rows with OBGPU_ENC_RAW forced on every column. A block in which a column would be stored as var-length cells (NULLs
 * dominate, ob_raw_encoder.cpp:106-110) is left to the host writer: its size reads 0.
 * ============================================================================================= */
typedef struct obgpu_encode_col {
  const int64_t *dev_vals;   /* [total_rows] value image of the datum (low type_store_size bytes are stored) */
  const uint8_t *dev_null;   /* [total_rows] 1 => NULL; NULL pointer: no NULL cell                           */
  int32_t obj_type;          /* OBGPU_OBJ_* (integer classes)                                                */
  int32_t byte_packing_only; /* 1 => ObMicroBlockEncoderOpt.enable_bit_packing_ == false                     */
} obgpu_encode_col;
typedef struct obgpu_encoded obgpu_encoded;
int obgpu_encode_columns(obgpu_ctx *ctx, const obgpu_encode_col *cols, int32_t n_cols, int32_t rowkey_col_cnt,
                         int64_t total_rows, int64_t rows_per_block, int32_t align, obgpu_encoded **out);
/* The same over a merge result: result_cols[i] = -1 the rowkey, -2, -3 ...: the following rowkey columns, >= 0 a payload
 * column (a column group of a column-oriented merge is one call with the group's columns: ObWriteHelper::project). */
int obgpu_merge_result_encode(obgpu_merge_result *res, const int32_t *result_cols, const int32_t *obj_types, int32_t n_cols,
                              int32_t rowkey_col_cnt, int64_t rows_per_block, int32_t align, obgpu_encoded **out);
/* The same with a codec per column. encodings[i]: OBGPU_ENC_RAW / _DICT / _RLE / _CONST / _INTEGER_BASE_DIFF (forced) or
 * OBGPU_ENC_AUTO (chosen per micro-block like obgpu_writer_encode_table's OBGPU_ENC_AUTO); encodings == NULL: every column RAW.
 * Byte for byte the host writer's blocks for the same rows and encodings. A block the host writer would encode differently
 * from the device reads size 0 and counts in n_host_blocks: RAW (forced or chosen) with var-stored cells, or a forced codec the
 * host writer refuses for the block's data (CONST with more than 32 exceptions or more than 10 % of the rows, DICT / RLE on a
 * column whose every cell is NULL); encode those blocks with the host writer and the same encodings.
 * INTEGER_BASE_DIFF over a single value is written as RAW, as the host writer does.
 * Call-level refusals: a string column -> OBGPU_NOT_SUPPORTED; an encoding outside the six -> OBGPU_INVALID_ARGUMENT; some
 * column not RAW and rows_per_block > 4096 (the codec kernel's cap) -> OBGPU_NOT_SUPPORTED; some column not RAW and the largest
 * block the requested codecs can write, plus the kernel's per-row scratch, does not fit one CTA's shared memory
 * -> OBGPU_NOT_SUPPORTED. Every column RAW runs the RAW encoder of obgpu_encode_columns. */
int obgpu_encode_columns_with(obgpu_ctx *ctx, const obgpu_encode_col *cols, const int32_t *encodings, int32_t n_cols,
                              int32_t rowkey_col_cnt, int64_t total_rows, int64_t rows_per_block, int32_t align, obgpu_encoded **out);
int obgpu_merge_result_encode_with(obgpu_merge_result *res, const int32_t *result_cols, const int32_t *obj_types,
                                   const int32_t *encodings, int32_t n_cols, int32_t rowkey_col_cnt, int64_t rows_per_block,
                                   int32_t align, obgpu_encoded **out);
typedef struct obgpu_encoded_info {
  int64_t image_size;    /* bytes of the image (aligned block slots)          */
  int64_t total_rows;
  int32_t n_blocks;
  int32_t n_host_blocks; /* blocks left to the host writer (size 0)           */
} obgpu_encoded_info;
int obgpu_encoded_get_info(obgpu_encoded *enc, obgpu_encoded_info *info);
/* Image + per block offset / size to host memory; any of the three may be NULL. */
int obgpu_encoded_fetch(obgpu_encoded *enc, void *host_image, int64_t image_cap, int64_t *host_offsets, int64_t *host_sizes,
                        int32_t blocks_cap);
/* The device image itself (valid until obgpu_encoded_free), e.g. to re-open it as a page batch without a host round trip. */
int obgpu_encoded_device_image(obgpu_encoded *enc, const void **dev_image, const int64_t **dev_offsets, const uint32_t **dev_sizes);
/* Column checksums (K16) of the encoded rows, n_cols values in host memory. */
int obgpu_encoded_column_checksums(obgpu_encoded *enc, int64_t *host_checksums);
void obgpu_encoded_free(obgpu_encoded *enc);
/* Column checksums of plain device columns (no encode). */
int obgpu_column_checksums(obgpu_ctx *ctx, const obgpu_encode_col *cols, int32_t n_cols, int64_t total_rows, int64_t *host_checksums);

#ifdef __cplusplus
}
#endif
#endif /* OBGPU_COMPACTION_H_ */
