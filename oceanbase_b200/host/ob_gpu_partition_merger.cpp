#include "ob_gpu_partition_merger.h"

#include <algorithm>

namespace oceanbase {
namespace compaction {
using namespace common;

ObGpuPartitionMajorMerger::~ObGpuPartitionMajorMerger() { reset(); }

void ObGpuPartitionMajorMerger::reset() {
  if (result_) obgpu_merge_result_free(result_);
  result_ = nullptr;
  for (obgpu_batch *b : batches_) obgpu_batch_close(b);
  batches_.clear();
  if (ctx_) obgpu_ctx_destroy(ctx_);
  ctx_ = nullptr;
  merged_ = false;
  cursor_ = 0;
  info_ = obgpu_merge_info{};
}

int ObGpuPartitionMajorMerger::init(int device, const std::vector<ObGpuMergeTable> &tables, const ObGpuMergeSchema &schema) {
  int ret = OB_SUCCESS;
  if (ctx_ != nullptr) {
    ret = OB_INIT_TWICE;
  } else if (tables.empty() || (!schema.default_vals_.empty() && schema.default_vals_.size() != schema.payload_cols_.size()) ||
             (!schema.default_null_.empty() && schema.default_null_.size() != schema.payload_cols_.size()) ||
             (!schema.payload_is_string_.empty() && schema.payload_is_string_.size() != schema.payload_cols_.size()) ||
             schema.more_rowkey_cols_.size() + 1 > OBGPU_MERGE_MAX_KEY_COLS) {
    ret = OB_INVALID_ARGUMENT;
  } else if (OB_SUCCESS != obgpu_ctx_create(device, &ctx_)) {
    ctx_ = nullptr;
    ret = OB_NOT_SUPPORTED;  // no device: the caller keeps ObPartitionMajorMerger
  } else {
    schema_ = schema;
    for (size_t i = 0; OB_SUCCESS == ret && i < tables.size(); ++i) {
      const ObGpuMergeTable &t = tables[i];
      obgpu_batch *b = nullptr;
      ret = obgpu_batch_open(ctx_, t.image_, t.image_size_, t.offsets_, t.sizes_, t.block_count_, 0, nullptr, &b);
      if (OB_SUCCESS == ret) batches_.push_back(b);
    }
    if (OB_SUCCESS != ret) reset();
  }
  return ret;
}

int ObGpuPartitionMajorMerger::merge_partition() {
  int ret = OB_SUCCESS;
  if (ctx_ == nullptr) {
    ret = OB_NOT_INIT;
  } else if (merged_) {
    ret = OB_ERR_UNEXPECTED;
  } else {
    std::vector<int32_t> keys(1, schema_.rowkey_col_);
    keys.insert(keys.end(), schema_.more_rowkey_cols_.begin(), schema_.more_rowkey_cols_.end());
    ret = obgpu_merge_runs_keys(ctx_, batches_.data(), (int32_t)batches_.size(), keys.data(), (int32_t)keys.size(), schema_.flag_col_,
                                schema_.payload_cols_.data(), (int32_t)schema_.payload_cols_.size(),
                                schema_.default_vals_.empty() ? nullptr : schema_.default_vals_.data(),
                                schema_.default_null_.empty() ? nullptr : schema_.default_null_.data(), &result_);
    if (OB_SUCCESS == ret) ret = obgpu_merge_result_info(result_, &info_);
    if (OB_SUCCESS == ret) merged_ = true;
  }
  return ret;
}

int ObGpuPartitionMajorMerger::get_next_rows(int64_t max_rows, ObGpuMergedRows &rows) {
  int ret = OB_SUCCESS;
  if (!merged_) {
    ret = OB_NOT_INIT;
  } else if (max_rows <= 0) {
    ret = OB_INVALID_ARGUMENT;
  } else if (cursor_ >= info_.out_rows) {
    rows.row_count_ = 0;
    ret = OB_ITER_END;
  } else {
    const int64_t n = std::min(max_rows, info_.out_rows - cursor_);
    const size_t nc = schema_.payload_cols_.size();
    rows.row_count_ = n;
    rows.rowkeys_.resize((size_t)n);
    rows.values_.resize(nc);
    rows.nulls_.resize(nc);
    rows.heap_.assign(nc, {});
    rows.offsets_.assign(nc, {});
    rows.more_rowkeys_.resize(schema_.more_rowkey_cols_.size());
    ret = obgpu_merge_result_fetch(result_, -1, cursor_, n, rows.rowkeys_.data(), nullptr);
    for (size_t k = 0; OB_SUCCESS == ret && k < rows.more_rowkeys_.size(); ++k) {
      rows.more_rowkeys_[k].resize((size_t)n);
      ret = obgpu_merge_result_fetch(result_, -2 - (int32_t)k, cursor_, n, rows.more_rowkeys_[k].data(), nullptr);
    }
    for (size_t c = 0; OB_SUCCESS == ret && c < nc; ++c) {
      rows.values_[c].assign((size_t)n, 0);
      rows.nulls_[c].resize((size_t)n);
      if (!schema_.payload_is_string_.empty() && schema_.payload_is_string_[c]) {
        // references -> bytes for this window only (the writer consumes ObString cells)
        rows.offsets_[c].resize((size_t)n + 1);
        int64_t need = 0;
        ret = obgpu_merge_result_fetch_strings(result_, (int32_t)c, cursor_, n, nullptr, 0, rows.offsets_[c].data(),
                                               rows.nulls_[c].data(), &need);
        if (OBGPU_BUF_NOT_ENOUGH == ret || (OB_SUCCESS == ret && need > 0)) {
          rows.heap_[c].resize((size_t)need);
          ret = obgpu_merge_result_fetch_strings(result_, (int32_t)c, cursor_, n, rows.heap_[c].data(), need,
                                                 rows.offsets_[c].data(), rows.nulls_[c].data(), &need);
        }
      } else {
        ret = obgpu_merge_result_fetch(result_, (int32_t)c, cursor_, n, rows.values_[c].data(), rows.nulls_[c].data());
      }
    }
    if (OB_SUCCESS == ret) cursor_ += n;
  }
  return ret;
}

int ObGpuPartitionMajorMerger::write_column_groups(const std::vector<ObGpuColumnGroup> &groups, int64_t rows_per_block, int32_t align,
                                                   std::vector<ObGpuEncodedColumnGroup> &out) {
  int ret = OB_SUCCESS;
  if (!merged_) {
    ret = OB_NOT_INIT;
  } else if (groups.empty() || rows_per_block <= 0 || info_.out_rows <= 0) {
    ret = OB_INVALID_ARGUMENT;
  }
  out.clear();
  out.resize(OB_SUCCESS == ret ? groups.size() : 0);
  // every group is enqueued before the first one is fetched: the encodes run back to back on the ctx stream
  std::vector<obgpu_encoded *> enc(groups.size(), nullptr);
  for (size_t g = 0; OB_SUCCESS == ret && g < groups.size(); ++g) {
    const ObGpuColumnGroup &cg = groups[g];
    if (cg.cols_.empty() || cg.cols_.size() != cg.obj_types_.size() || (!cg.encodings_.empty() && cg.encodings_.size() != cg.cols_.size()))
      ret = OB_INVALID_ARGUMENT;
    else ret = obgpu_merge_result_encode_with(result_, cg.cols_.data(), cg.obj_types_.data(), cg.encodings_.empty() ? nullptr : cg.encodings_.data(),
                                              (int32_t)cg.cols_.size(), cg.rowkey_col_cnt_, rows_per_block, align, &enc[g]);
  }
  for (size_t g = 0; OB_SUCCESS == ret && g < groups.size(); ++g) {
    const ObGpuColumnGroup &cg = groups[g];
    ObGpuEncodedColumnGroup &o = out[g];
    obgpu_encoded_info info{};
    ret = obgpu_encoded_get_info(enc[g], &info);
    if (OB_SUCCESS != ret) break;
    o.row_count_ = info.total_rows;
    o.host_encoded_blocks_ = info.n_host_blocks;
    o.offsets_.resize((size_t)info.n_blocks);
    o.sizes_.resize((size_t)info.n_blocks);
    o.image_.resize((size_t)info.image_size);
    o.column_checksums_.resize(cg.cols_.size());
    ret = obgpu_encoded_fetch(enc[g], o.image_.data(), info.image_size, o.offsets_.data(), o.sizes_.data(), info.n_blocks);
    if (OB_SUCCESS == ret) ret = obgpu_encoded_column_checksums(enc[g], o.column_checksums_.data());
    if (OB_SUCCESS == ret && info.n_host_blocks > 0) {
      // the blocks the device left out (ObRawEncoder stores a NULL-dominated column as var-length cells, or a forced codec the
      // block's data does not take): their rows come back as rows and go through the host writer with the same encodings; the
      // image is laid out again with them in place
      std::vector<uint8_t> image;
      std::vector<int64_t> offsets((size_t)info.n_blocks);
      std::vector<int64_t> vals;
      std::vector<uint8_t> nulls;
      for (int32_t b = 0; OB_SUCCESS == ret && b < info.n_blocks; ++b) {
        const size_t at = image.size();
        offsets[(size_t)b] = (int64_t)at;
        if (o.sizes_[(size_t)b] != 0) {
          image.insert(image.end(), o.image_.begin() + o.offsets_[(size_t)b], o.image_.begin() + o.offsets_[(size_t)b] + o.sizes_[(size_t)b]);
        } else {
          const int64_t row0 = (int64_t)b * rows_per_block, n = std::min(rows_per_block, info.total_rows - row0);
          const size_t nc = cg.cols_.size();
          vals.assign(nc * (size_t)n, 0);
          nulls.assign(nc * (size_t)n, 0);
          std::vector<obgpu_col_input> in(nc);
          for (size_t c = 0; OB_SUCCESS == ret && c < nc; ++c) {
            ret = obgpu_merge_result_fetch(result_, cg.cols_[c], row0, n, vals.data() + c * (size_t)n,
                                           cg.cols_[c] >= 0 ? nulls.data() + c * (size_t)n : nullptr);
            in[c] = obgpu_col_input{};
            in[c].obj_type = cg.obj_types_[c];
            in[c].encoding = cg.encodings_.empty() ? OBGPU_ENC_RAW : cg.encodings_[c];
            in[c].i64 = vals.data() + c * (size_t)n;
            in[c].is_null = nulls.data() + c * (size_t)n;
          }
          if (OB_SUCCESS == ret) {
            const int64_t bound = obgpu_writer_block_bound(in.data(), (int32_t)nc, 0, n);
            image.resize(at + (size_t)bound);
            int64_t sz = 0;
            ret = obgpu_writer_encode_block(in.data(), (int32_t)nc, cg.rowkey_col_cnt_, 0, n, image.data() + at, bound, &sz);
            if (OB_SUCCESS == ret) { image.resize(at + (size_t)sz); o.sizes_[(size_t)b] = sz; }
          }
        }
        image.resize((image.size() + (size_t)align - 1) / (size_t)align * (size_t)align, 0);
      }
      if (OB_SUCCESS == ret) { o.image_.swap(image); o.offsets_.swap(offsets); }
    }
  }
  for (obgpu_encoded *e : enc) obgpu_encoded_free(e);
  if (OB_SUCCESS != ret) out.clear();
  return ret;
}

}  // namespace compaction
}  // namespace oceanbase
