// C++ parity test of ObGpuPartitionMajorMerger::write_column_groups with per-column encodings (ObGpuColumnGroup::encodings_):
// two encoded runs are merged on the device, and every column group written with OBGPU_ENC_AUTO (one group also with a
// NULL-dominated RAW column, whose blocks the device leaves to the host writer) must equal, block by block, the host writer's
// image of the oracle's merged rows (oracle/ob_oracle.c: ora_major_merge) with the same encodings, pass the oracle's checksum
// checks and carry the oracle's column checksums. Exit 77 without a device.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../oceanbase_b200/host/ob_gpu_partition_merger.h"
extern "C" {
#include "../../include/obgpu_writer.h"
#include "../../oracle/ob_oracle.h"
}

using namespace oceanbase;
using namespace oceanbase::common;
using namespace oceanbase::compaction;

static int g_fail = 0;
#define ASSERT_EQ(a, b)                                                                           \
  do {                                                                                            \
    const long long va__ = (long long)(a), vb__ = (long long)(b);                                 \
    if (va__ != vb__) {                                                                           \
      printf("FAIL %s:%d  %s = %lld, expected %lld\n", __FILE__, __LINE__, #a, va__, vb__);       \
      ++g_fail;                                                                                   \
    }                                                                                             \
  } while (0)

static uint64_t mix(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

struct Run {
  std::vector<int64_t> key, flag;
  std::vector<std::vector<int64_t>> vals;   // [3]
  std::vector<std::vector<uint8_t>> ext;    // [3]: 0 value, 1 NULL
  std::vector<uint8_t> image;
  std::vector<int64_t> offsets, sizes;
};

static void encode(Run &r, int64_t rows_per_block) {
  const int64_t n = (int64_t)r.key.size();
  obgpu_col_input cols[5];
  memset(cols, 0, sizeof(cols));
  cols[0].obj_type = OBGPU_OBJ_INT; cols[0].encoding = OBGPU_ENC_INTEGER_BASE_DIFF; cols[0].i64 = r.key.data();
  cols[1].obj_type = OBGPU_OBJ_TINYINT; cols[1].encoding = OBGPU_ENC_RAW; cols[1].i64 = r.flag.data();
  for (int c = 0; c < 3; ++c) {
    cols[2 + c].obj_type = OBGPU_OBJ_INT; cols[2 + c].encoding = OBGPU_ENC_AUTO;
    cols[2 + c].i64 = r.vals[c].data(); cols[2 + c].is_null = r.ext[c].data();
  }
  obgpu_table_image *img = nullptr;
  if (obgpu_writer_encode_table(cols, 5, 1, n, rows_per_block, 128, 2, &img) != 0) { printf("encode failed\n"); exit(2); }
  int64_t size = 0; int32_t nb = 0;
  obgpu_table_image_info(img, &size, &nb);
  r.image.assign((size_t)size + 64, 0);
  r.offsets.resize((size_t)nb); r.sizes.resize((size_t)nb);
  obgpu_table_image_export(img, r.image.data(), size, r.offsets.data(), r.sizes.data(), nb);
  obgpu_table_image_free(img);
}

int main() {
  {
    obgpu_ctx *probe = nullptr;
    if (obgpu_ctx_create(0, &probe) != 0) { printf("no CUDA device: the adapter refuses (no CPU fallback)\n"); return 77; }
    obgpu_ctx_destroy(probe);
  }
  // payload: 0 low-cardinality, 1 NULL in 60 % of the rows with 60-bit values, 2 runs of 50 rows; disjoint rowkeys
  std::vector<Run> runs(2);
  for (int r = 0; r < 2; ++r) {
    Run &run = runs[r];
    run.vals.assign(3, {}); run.ext.assign(3, {});
    for (int64_t i = 0; i < 6000; ++i) {
      const uint64_t h = mix((uint64_t)i * 131u + (uint64_t)r);
      if (h % 4 == 0) continue;
      run.key.push_back(1000 + i * 2 + r);
      run.flag.push_back(OBGPU_DF_INSERT);
      const uint64_t h1 = mix(h + 977u);
      run.vals[0].push_back((int64_t)(h % 8) * 1000003);
      run.ext[0].push_back(0);
      run.vals[1].push_back(h1 % 100 < 60 ? 0 : (int64_t)(h1 >> 4));
      run.ext[1].push_back(h1 % 100 < 60 ? 1 : 0);
      run.vals[2].push_back((int64_t)mix((uint64_t)(i / 50)) >> 20);
      run.ext[2].push_back(0);
    }
    encode(run, 800);
  }
  std::vector<ObGpuMergeTable> tables;
  for (Run &r : runs) {
    ObGpuMergeTable t;
    t.image_ = r.image.data(); t.image_size_ = (int64_t)r.image.size() - 64;
    t.offsets_ = r.offsets.data(); t.sizes_ = r.sizes.data(); t.block_count_ = (int32_t)r.offsets.size();
    tables.push_back(t);
  }
  ObGpuMergeSchema schema;
  schema.rowkey_col_ = 0; schema.flag_col_ = 1; schema.payload_cols_ = {2, 3, 4};
  ObGpuPartitionMajorMerger merger;
  ASSERT_EQ(merger.init(0, tables, schema), OB_SUCCESS);
  ASSERT_EQ(merger.merge_partition(), OB_SUCCESS);
  // the oracle's merged rows
  std::vector<ora_merge_run> oruns(runs.size());
  std::vector<std::vector<uint8_t>> flag8(runs.size());
  std::vector<std::vector<const int64_t *>> vp(runs.size());
  std::vector<std::vector<const uint8_t *>> ep(runs.size());
  int64_t total = 0;
  for (size_t i = 0; i < runs.size(); ++i) {
    flag8[i].assign(runs[i].flag.begin(), runs[i].flag.end());
    for (int c = 0; c < 3; ++c) { vp[i].push_back(runs[i].vals[c].data()); ep[i].push_back(runs[i].ext[c].data()); }
    oruns[i].n = (int64_t)runs[i].key.size(); oruns[i].key = runs[i].key.data(); oruns[i].flag = flag8[i].data();
    oruns[i].vals = vp[i].data(); oruns[i].ext = ep[i].data();
    total += oruns[i].n;
  }
  std::vector<int64_t> okey((size_t)total + 1);
  std::vector<std::vector<int64_t>> ov(3, std::vector<int64_t>((size_t)total + 1));
  std::vector<std::vector<uint8_t>> on(3, std::vector<uint8_t>((size_t)total + 1));
  int64_t *ovp[3] = {ov[0].data(), ov[1].data(), ov[2].data()};
  uint8_t *onp[3] = {on[0].data(), on[1].data(), on[2].data()};
  int64_t orows = 0, stats[2] = {0, 0};
  ASSERT_EQ(ora_major_merge(oruns.data(), (int32_t)runs.size(), 3, nullptr, nullptr, total, okey.data(), ovp, onp, &orows, stats), 0);
  ASSERT_EQ(merger.get_output_row_count(), orows);

  std::vector<ObGpuColumnGroup> groups(3);
  groups[0].cols_ = {-1, 0, 1, 2}; groups[0].obj_types_.assign(4, OBGPU_OBJ_INT); groups[0].rowkey_col_cnt_ = 1;
  groups[0].encodings_ = {OBGPU_ENC_AUTO, OBGPU_ENC_AUTO, OBGPU_ENC_RAW, OBGPU_ENC_AUTO};   // column 1 RAW: var-stored -> host writer
  groups[1].cols_ = {0}; groups[1].obj_types_ = {OBGPU_OBJ_INT}; groups[1].encodings_ = {OBGPU_ENC_AUTO};
  groups[2].cols_ = {2, 1}; groups[2].obj_types_.assign(2, OBGPU_OBJ_INT); groups[2].encodings_.assign(2, OBGPU_ENC_AUTO);
  std::vector<ObGpuEncodedColumnGroup> enc;
  const int64_t rpb = 700;
  ASSERT_EQ(merger.write_column_groups(groups, rpb, 128, enc), OB_SUCCESS);
  ASSERT_EQ((long long)enc.size(), 3);
  for (size_t g = 0; g < enc.size() && g_fail < 10; ++g) {
    const ObGpuColumnGroup &cg = groups[g];
    std::vector<obgpu_col_input> in(cg.cols_.size());
    for (size_t c = 0; c < cg.cols_.size(); ++c) {
      memset(&in[c], 0, sizeof(in[c]));
      in[c].obj_type = OBGPU_OBJ_INT; in[c].encoding = cg.encodings_[c];
      in[c].i64 = cg.cols_[c] < 0 ? okey.data() : ov[(size_t)cg.cols_[c]].data();
      in[c].is_null = cg.cols_[c] < 0 ? nullptr : on[(size_t)cg.cols_[c]].data();
      ASSERT_EQ(enc[g].column_checksums_[c], ora_column_checksum(in[c].i64, in[c].is_null, orows, 8));
    }
    obgpu_table_image *img = nullptr;
    ASSERT_EQ(obgpu_writer_encode_table(in.data(), (int32_t)in.size(), cg.rowkey_col_cnt_, orows, rpb, 128, 2, &img), 0);
    int64_t size = 0; int32_t nb = 0;
    obgpu_table_image_info(img, &size, &nb);
    std::vector<uint8_t> want((size_t)size);
    std::vector<int64_t> woff((size_t)nb), wsz((size_t)nb);
    obgpu_table_image_export(img, want.data(), size, woff.data(), wsz.data(), nb);
    obgpu_table_image_free(img);
    if (g == 0) ASSERT_EQ(enc[g].host_encoded_blocks_ > 0, 1);
    else ASSERT_EQ(enc[g].host_encoded_blocks_, 0);
    ASSERT_EQ(enc[g].row_count_, orows);
    ASSERT_EQ((long long)enc[g].offsets_.size(), nb);
    ASSERT_EQ((long long)enc[g].image_.size(), size);
    int kinds = 0;
    for (int32_t b = 0; b < nb && g_fail < 10; ++b) {
      ASSERT_EQ(enc[g].offsets_[(size_t)b], woff[(size_t)b]);
      ASSERT_EQ(enc[g].sizes_[(size_t)b], wsz[(size_t)b]);
      if (enc[g].sizes_[(size_t)b] == wsz[(size_t)b] && enc[g].offsets_[(size_t)b] == woff[(size_t)b])
        ASSERT_EQ(memcmp(enc[g].image_.data() + woff[(size_t)b], want.data() + woff[(size_t)b], (size_t)wsz[(size_t)b]), 0);
      ora_block blk;
      ASSERT_EQ(ora_block_init(&blk, enc[g].image_.data() + enc[g].offsets_[(size_t)b], enc[g].sizes_[(size_t)b]), 0);
      ASSERT_EQ(ora_block_verify_checksums(&blk), 0);
      for (size_t c = 0; c < cg.cols_.size(); ++c) kinds |= 1 << want[(size_t)woff[(size_t)b] + 64 + 16 * c + 1];
    }
    ASSERT_EQ(kinds != (1 << 0), 1);   // not every column RAW
  }
  if (g_fail) { printf("%d failures\n", g_fail); return 1; }
  printf("partition merger codec tests passed\n");
  return 0;
}
