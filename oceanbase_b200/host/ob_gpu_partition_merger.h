// ob_gpu_partition_merger.h -- host-side (C++) adapter for the major-compaction merge, written the way a
// maintainer would add it next to compaction/ob_partition_merger.h: the names and call order mirror
// ObPartitionMajorMerger (merge_partition -> rows handed to the macro block writer), the work goes through
// the C-ABI in include/obgpu_compaction.h. Stand-ins for reference types are minimal and local.
#ifndef OB_GPU_PARTITION_MERGER_H_
#define OB_GPU_PARTITION_MERGER_H_

#include <cstdint>
#include <vector>

extern "C" {
#include "../../include/obgpu_compaction.h"
#include "../../include/obgpu_writer.h"
}
#include "ob_gpu_micro_block_decoder.h"

namespace oceanbase {
namespace compaction {

// One table of the merge (ObTablesHandleArray entry): the encoded micro blocks of the merge range.
struct ObGpuMergeTable {
  const void *image_ = nullptr;
  int64_t image_size_ = 0;
  const int64_t *offsets_ = nullptr;
  const int64_t *sizes_ = nullptr;
  int32_t block_count_ = 0;
};

// Column roles inside the tables' row layout (ObStaticMergeParam / ObTableReadInfo would provide them).
struct ObGpuMergeSchema {
  int32_t rowkey_col_ = 0;              // first (or only) rowkey column
  std::vector<int32_t> more_rowkey_cols_;  // the following columns of a composite rowkey, in comparison order
  int32_t flag_col_ = -1;               // column holding the ObDmlFlag image, -1: every row DF_INSERT
  std::vector<int32_t> payload_cols_;
  std::vector<uint8_t> payload_is_string_;  // per payload column: 1 => VARCHAR / CHAR (empty: all integer class)
  std::vector<int64_t> default_vals_;   // default row (ObMajorPartitionMergeFuser::default_row_)
  std::vector<uint8_t> default_null_;   // empty: every default is NULL
};

// Window of the merged row stream, what ObPartitionMajorMerger::process hands to
// ObMacroBlockWriter::append_row row by row (here: column arrays for append_batch).
struct ObGpuMergedRows {
  int64_t row_count_ = 0;
  std::vector<int64_t> rowkeys_;
  std::vector<std::vector<int64_t>> more_rowkeys_;  // [extra rowkey column][row]
  std::vector<std::vector<int64_t>> values_;   // [payload column][row] (integer class)
  std::vector<std::vector<uint8_t>> nulls_;    // 1 => NULL
  // string payload columns: cell i of column c = heap_[c][offsets_[c][i] .. offsets_[c][i + 1])
  std::vector<std::vector<char>> heap_;
  std::vector<std::vector<int64_t>> offsets_;
};

// One column group of a column-oriented merge (ObStorageColumnGroupSchema): which columns of the merged row it stores, in
// row order of the group. -1 = the rowkey, -2, -3 ... = the following rowkey columns, >= 0 = payload column index.
struct ObGpuColumnGroup {
  std::vector<int32_t> cols_;
  std::vector<int32_t> obj_types_;   // OBGPU_OBJ_* of every column (integer classes)
  int32_t rowkey_col_cnt_ = 0;       // > 0 for the group that carries the rowkey (all-column / rowkey group)
  // OBGPU_ENC_RAW / _DICT / _RLE / _CONST / _INTEGER_BASE_DIFF / _AUTO of every column; empty: every column RAW
  std::vector<int32_t> encodings_;
};

// What the writer of one column group produced: the micro-blocks of its SSTable + the column checksums of its rows.
struct ObGpuEncodedColumnGroup {
  std::vector<uint8_t> image_;
  std::vector<int64_t> offsets_, sizes_;
  std::vector<int64_t> column_checksums_;
  int64_t row_count_ = 0;
  int32_t host_encoded_blocks_ = 0;  // blocks the device left to the host writer (var-stored RAW cells, a codec refused for the block)
};

class ObGpuPartitionMajorMerger {
public:
  ObGpuPartitionMajorMerger() = default;
  ~ObGpuPartitionMajorMerger();
  ObGpuPartitionMajorMerger(const ObGpuPartitionMajorMerger &) = delete;
  ObGpuPartitionMajorMerger &operator=(const ObGpuPartitionMajorMerger &) = delete;

  // tables oldest -> newest (tables_handle order); returns OB_NOT_SUPPORTED when no device is usable so that
  // the caller keeps the CPU merger.
  int init(int device, const std::vector<ObGpuMergeTable> &tables, const ObGpuMergeSchema &schema);
  // ObPartitionMajorMerger::merge_partition: runs the whole merge of the range on the device.
  int merge_partition();
  int64_t get_output_row_count() const { return info_.out_rows; }
  int64_t get_dropped_delete_count() const { return info_.dropped_deletes; }
  int64_t get_fused_row_count() const { return info_.fused_rows; }
  // Next window of at most max_rows merged rows in rowkey order; OB_ITER_END after the last one.
  int get_next_rows(int64_t max_rows, ObGpuMergedRows &rows);
  // Column-oriented merge, writer side (ObCOMergeLogReplayer::replay_merge_log -> ObCOMergeWriter::replay_mergelog ->
  // ObWriteHelper::project / append, column_store/ob_column_oriented_merger.cpp:722-745, ob_co_merge_writer.cpp:67-117,345):
  // the merged stream -- produced once by merge_partition -- is replayed into the writer of every column group. Here a
  // writer is the device encoder (obgpu_merge_result_encode_with): the rows never leave the device as rows, each group comes
  // back as reference-format micro-blocks (the group's encodings_, RAW when empty) + its column checksums. rows_per_block cuts
  // the blocks; a block the device leaves out is encoded by the host writer with the same encodings and spliced in.
  int write_column_groups(const std::vector<ObGpuColumnGroup> &groups, int64_t rows_per_block, int32_t align,
                          std::vector<ObGpuEncodedColumnGroup> &out);
  void reset();

private:
  obgpu_ctx *ctx_ = nullptr;
  std::vector<obgpu_batch *> batches_;
  ObGpuMergeSchema schema_;
  obgpu_merge_result *result_ = nullptr;
  obgpu_merge_info info_{};
  int64_t cursor_ = 0;
  bool merged_ = false;
};

}  // namespace compaction
}  // namespace oceanbase
#endif
