// libobgpu_scan.so -- micro-block scan kernels (sm_100a) and the C-ABI around them.
//
// A page batch (thousands of ~16 KiB micro-blocks, PAX or CS format) is scanned by
//   index   (once, at batch open): one thread per (block, column) -> 96-byte decode plan + block record
//   count   : one warp per block; filter columns staged with coalesced 16-byte loads; white-filter tree,
//             predicate-on-dictionary for dictionary-coded columns, warp ballot / SIMD-in-register
//             compares -> packed selection bitmap + per-block count (K4/K6/K9/K14)
//   prefix  : exclusive scan of the counts -> dense output offset of every block
//   project : one CTA per block; TMA bulk copy (cp.async.bulk + mbarrier) of the block or of the projected
//             column regions into shared memory; bitmap -> ascending selected-row list; columns
//             distributed over the warps, coalesced 8-byte stores into the dense VEC_FIXED /
//             VEC_DISCRETE buffers (K1-K8); sparse selections are decoded straight from global memory
//   aggregate (optional): COUNT / SUM / SUM(a*b) / MIN / MAX over the dense columns, 128-bit exact
// and merge_kernels.cuh (included at the end) holds the major-compaction merge.
//
// Reference control flow this replaces (per block, per <=256-row batch, per column virtual calls):
//   ObIMicroBlockRowScanner::apply_filter        blocksstable/ob_micro_block_row_scanner.cpp:361,927
//   ObPushdownFilterExecutor::execute            sql/engine/basic/ob_pushdown_filter.cpp:1551-1624
//   ObMicroBlockDecoder::filter_pushdown_filter  encoding/ob_micro_block_decoder.cpp:1680-1755
//   ObBitmap::get_row_ids                        deps/oblib/src/lib/container/ob_bitmap.cpp:540
//   ObMicroBlockDecoder::get_rows                encoding/ob_micro_block_decoder.cpp:2473-2544
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/obgpu_scan.h"
#include "../../include/obgpu_skip_index.h"
#include "ob_format.h"
#include "scan_device.cuh"

using namespace obdev;

// =================================================================================================
// Kernel parameter block
// =================================================================================================
struct FilterNodeDev {
  int8_t kind;
  int8_t slot;        // dictionary-bitset slot of a leaf (-1: none)
  int8_t range_ok;    // leaf: integer compare reducible to one range test on the 64-bit image
  int8_t negate;      // leaf: NE = NOT(range) for non-NULL rows
  int16_t used_idx;   // leaf: index into ScanParams::used_col
  int16_t op;
  int16_t param_begin;
  int16_t n_params;
  int16_t n_children;
  int16_t pad;
  uint64_t lo;        // range test: (uint64)(v - lo) <= span
  uint64_t span;
};

// String-equality leaves (EQ / NE / IN): slot of a (length, first 8 bytes) pair in a 64-slot hash. When one of the multipliers
// maps the leaf's constants to distinct slots (FilterNodeDev::pad = multiplier index + 1), the constants are stored in slot
// order and FilterNodeDev::span is the occupancy mask: a dictionary entry finds the ONLY constant it can equal with one
// popcount instead of walking the list.
__host__ __device__ __forceinline__ uint32_t str_eq_slot(uint64_t pre, uint32_t len, int m) {
  const uint64_t mult = 0xD6E8FEB86659FD93ull + 2ull * (uint64_t)m * 0x9E3779B97F4A7C15ull;   // odd
  return (uint32_t)(((pre ^ ((uint64_t)len * 0x9E3779B97F4A7C15ull)) * mult) >> 58);
}
constexpr int kStrEqHashTries = 8;

struct ParamDev {
  int64_t i64;
  uint32_t heap_off;
  uint32_t len;
};

constexpr int kParamHeap = 768;

// layout of obcs::XformRec (stream_codecs.cuh), declared here for the kernel parameter block
struct XformRecFwd { uint64_t orig_off; int64_t str_delta; };


struct ScanParams {
  const uint8_t *image;
  const uint64_t *blk_off;    // [n_blocks] byte offset of block i in image
  const uint32_t *blk_size;   // [n_blocks] exact block size
  const int64_t *bm_word_off; // [n_blocks + 1] prefix of ceil(rows / 32)
  int32_t n_blocks;
  const ColDesc *plans;       // [n_blocks][max_cols] decode plans built once at batch open (index kernel)
  const uint32_t *rows;       // [n_blocks] row counts (0: corrupt block)
  const BlockRec *recs;       // [n_blocks] addressing + header fields (index kernel)
  uint32_t *counts;           // [n_blocks] selected rows per block (count kernel)
  int32_t max_cols;
  int32_t n_used;
  int32_t used_col[kMaxUsedCols];
  uint8_t used_in_filter[kMaxUsedCols];
  uint8_t used_in_proj[kMaxUsedCols];
  int8_t used_rle_slot[kMaxUsedCols];  // run-table slot of a used column (-1: never RLE)
  int32_t n_nodes;
  int32_t simple_shape;       // 1: single leaf or AND over leaves only, 2: OR over leaves only, 0: generic
  FilterNodeDev nodes[kMaxNodes];
  ParamDev params[kMaxParams];
  alignas(8) uint8_t param_heap[kParamHeap];  // string constants, each 8-byte aligned and padded
  int32_t n_slots;
  int32_t bitset_words;       // words per slot
  int32_t n_rle_slots;
  int32_t rle_runs_cap;       // run-table capacity (runs) per slot
  int32_t n_proj;
  int32_t want_row_ids;
  int16_t proj_used[kMaxProj];
  void *out_data[kMaxProj];
  int32_t *out_lens[kMaxProj];
  uint32_t *out_nulls[kMaxProj];
  int32_t *has_null;          // [kMaxProj]
  uint64_t string_base;
  uint32_t *bitmap_words;
  int64_t *sel_offset;        // [n_blocks + 1]
  int32_t *row_ids;
  int32_t *status;
  int64_t out_cap;
  // skip index verdicts (nullptr: no aggregate rows attached): per block 0 uncertain / 1 always true / 2 always false,
  // and the same per (block, filter node)
  const uint8_t *blk_const;
  const uint8_t *leaf_const;
  // blocks of a batch whose CS streams were restated as RAW at open (stream_codecs.cuh): where each block came from
  const struct XformRecFwd *xf;
  // ---- shared-memory layout (bytes from the dynamic smem base) -------------------------------------
  // single-block kernels: [block][bitsets][rle tables][descs]
  // scan kernel:          [stage 0..kStages-1][bitsets][scratch 0][scratch 1], scratch = sel|bm|wpre|rle|descs
  uint32_t stage_bytes;       // scan kernel: bytes per stage buffer
  uint32_t smem_bitset;
  uint32_t smem_rle, smem_desc;            // single-block kernels
  uint32_t smem_scratch, scratch_bytes;    // project kernel
  uint32_t cw_desc, cw_bm, cw_bitset, cw_stage, cw_stage_bytes, cw_bytes;  // count kernel, per-warp: descs | bm | bitsets | stage
  uint32_t pw_rle, pw_rvals, pw_bytes;  // project kernel, per-warp region at off_desc: run values (u64) | RLE run table
  uint32_t off_plans;                   // project kernel: the block's n_proj decode plans (ColDesc), prefetched
  int32_t compact;                      // project kernel stages only the projected columns' regions (packed)
  int32_t sparse_split;                 // selectivity hint <= 1/16: sparse blocks go to the warp-per-block kernel
  int32_t no_stage;                     // blocks do not fit shared memory: every block is decoded from global memory
  int32_t proj_tiles;                   // blocks walked by one CTA of the project kernel (1, or 8 with the sparse split)
  uint32_t off_sel, off_bm, off_wpre, off_rle, off_desc;  // inside one scratch
  uint32_t smem_total;
  // ---- small-block pipelined kernels (scan_small.cuh): warp per block, cp.async rings ----------------------------
  int32_t pipe_count, pipe_project;         // which of the two kernels this scan uses
  int32_t pf_n;                             // filter columns = used columns [0, pf_n)
  uint32_t pf_off[8], pf_span[8];           // count: offset / capacity of a filter column's region inside a region slot
  uint32_t pc_meta_bytes, pc_region_bytes;  // count: bytes per meta / region slot
  uint32_t pc_meta, pc_region, pc_bm, pc_bitset, pc_bar, pc_bytes;   // count: per-warp layout
  uint32_t pp_off[kMaxProj], pp_span[kMaxProj];              // project: offset / capacity of a column's ranges in a region slot
  uint32_t pp_meta_bytes, pp_region_bytes, pp_hdr_bytes, pp_bm_bytes, pp_list;
  uint32_t pp_meta, pp_region, pp_sel, pp_wscr, pp_bar, pp_bytes;    // project: per-warp layout
  uint32_t rle_slot_bytes;    // bytes per run-table slot: mask[words_cap] (u32) + pre[words_cap] (u16)
  uint32_t rows_cap, words_cap;
};

// =================================================================================================
// PTX helpers: mbarrier + TMA bulk copy, acquire/release descriptor access, named barriers
// =================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_inval(uint64_t *bar) {
  asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
      "@P1 bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// A team of threads cooperating on one block: the whole CTA (bar 0), a single warp (bar < 0) or a
// subset of warps on a named barrier (bar > 0).
struct Team {
  int tid, nthreads, warp, nwarps, lane, bar_id;
  __device__ __forceinline__ void sync() const {
    if (bar_id == 0) __syncthreads();
    else if (bar_id < 0) __syncwarp();  // a single warp working on its own block
    else asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "r"(nthreads) : "memory");
  }
  __device__ __forceinline__ bool sync_or(bool pred) const {
    if (bar_id == 0) return __syncthreads_or(pred) != 0;
    int r;
    asm volatile(
        "{\n\t.reg .pred p, q;\n\tsetp.ne.b32 p, %1, 0;\n\tbar.red.or.pred q, %2, %3, p;\n\tselp.b32 %0, 1, 0, q;\n\t}"
        : "=r"(r)
        : "r"((int)pred), "r"(bar_id), "r"(nthreads)
        : "memory");
    return r != 0;
  }
};

__device__ __forceinline__ Team cta_team() {
  Team t;
  t.tid = threadIdx.x;
  t.nthreads = kThreads;
  t.warp = threadIdx.x >> 5;
  t.nwarps = kWarps;
  t.lane = threadIdx.x & 31;
  t.bar_id = 0;
  return t;
}

// =================================================================================================
// Predicate evaluation
// =================================================================================================
__device__ __forceinline__ bool int_pred(const ScanParams &p, const FilterNodeDev &nd, const ColDesc &d,
                                         uint64_t v) {
  const int64_t a = cmp_image(d, v);
  if (nd.range_ok) return (((uint64_t)a - nd.lo) <= nd.span) != (nd.negate != 0);
  const bool sgn = d.sc == 1;
  auto cmp3 = [&](int64_t c) -> int {
    if (sgn) return a < c ? -1 : (a > c ? 1 : 0);
    const uint64_t ua = (uint64_t)a, uc = (uint64_t)c;
    return ua < uc ? -1 : (ua > uc ? 1 : 0);
  };
  const int op = nd.op;
  if (op <= OP_NE) return cmp_to_bool(op, cmp3(p.params[nd.param_begin].i64));
  if (op == OP_BT) return cmp3(p.params[nd.param_begin].i64) >= 0 && cmp3(p.params[nd.param_begin + 1].i64) <= 0;
  if (op == OP_IN) {
    for (int i = 0; i < nd.n_params; ++i)
      if (cmp3(p.params[nd.param_begin + i].i64) == 0) return true;
    return false;
  }
  return false;
}

__device__ __forceinline__ bool str_pred(const ScanParams &p, const FilterNodeDev &nd, const uint8_t *s,
                                         uint32_t cell, uint32_t len) {
  auto cmp3 = [&](int k) -> int {
    const ParamDev &pp = p.params[nd.param_begin + k];
    return str_cmp(s, cell, len, p.param_heap + pp.heap_off, pp.len);
  };
  const int op = nd.op;
  if (op == OP_EQ || op == OP_NE || op == OP_IN) {
    // equality tests: length and the first 8 bytes decide almost every pair without a byte loop
    const uint64_t pre = len ? ld_bits(s, cell * 8u, (len < 8u ? len : 8u) * 8u) : 0ull;
    bool hit = false;
    for (int k = 0; k < nd.n_params && !hit; ++k) {
      const ParamDev &pp = p.params[nd.param_begin + k];
      hit = pp.len == len && (uint64_t)pp.i64 == pre && (len <= 8u || cmp3(k) == 0);
    }
    return hit != (op == OP_NE);
  }
  if (op <= OP_NE) return cmp_to_bool(op, cmp3(0));
  if (op == OP_BT) return cmp3(0) >= 0 && cmp3(1) <= 0;
  return false;
}

// Address the string cells of block `tile` are reported at: string_base + the block's offset in the CALLER's image.
// In a batch restated at open (CS stream codecs) the block moved and its string area shifted: the record undoes both.
__device__ __forceinline__ uint64_t block_string_addr(const ScanParams &p, int tile, uint64_t off) {
  if (p.xf != nullptr) {
    const XformRecFwd x = p.xf[tile];
    return p.string_base + x.orig_off + (uint64_t)x.str_delta;
  }
  return p.string_base + off;
}

// Everything a team needs to know about the block it is working on.
struct BlockCtx {
  BlockView b;
  uint32_t sbit;             // 8 * shared-window address of the staged block (fast-path loads)
  const ColDesc *descs;
  const uint32_t *bitsets;
  const uint8_t *rle_base;   // run-table scratch
  uint32_t rle_slot_bytes, rle_starts_bytes;  // slot stride; offset of pre[] inside a slot (= 4 * words_cap)
  __device__ __forceinline__ RleTable rle_table(int slot) const {
    RleTable t;
    t.mask = reinterpret_cast<const uint32_t *>(rle_base + (uint32_t)slot * rle_slot_bytes);
    t.pre = reinterpret_cast<const uint16_t *>(rle_base + (uint32_t)slot * rle_slot_bytes + rle_starts_bytes);
    return t;
  }
};

// generic per-row leaf (any codec, any type)
__device__ __forceinline__ bool eval_leaf(const ScanParams &p, const BlockCtx &c, const FilterNodeDev &nd,
                                          uint32_t row) {
  const int op = nd.op;
  if (op == OP_FALSE) return false;
  if (op == OP_TRUE) return true;
  const ColDesc &d = c.descs[nd.used_idx];
  RleTable rt{};
  const RleTable *rtp = nullptr;
  if (d.kind == K_RLE && d.rle_slot >= 0) {
    rt = c.rle_table(d.rle_slot);
    rtp = &rt;
  }
  if (is_dict_kind(d)) {
    uint32_t ref = ref_of(c.b.s, d, rtp, row);
    if (ref > d.dict_count + 1) ref = d.dict_count + 1;
    return (c.bitsets[nd.slot * p.bitset_words + (ref >> 5)] >> (ref & 31)) & 1u;
  }
  bool is_null;
  if (d.sc == 5) {
    uint32_t cell, len;
    str_cell(c.b, d, rtp, row, cell, len, is_null);
    if (op == OP_NU) return is_null;
    if (op == OP_NN) return !is_null;
    return !is_null && str_pred(p, nd, c.b.s, cell, len);
  }
  const uint64_t v = int_cell(c.b, d, rtp, row, is_null);
  if (op == OP_NU) return is_null;
  if (op == OP_NN) return !is_null;
  return !is_null && int_pred(p, nd, d, v);
}

__device__ __forceinline__ bool eval_tree(const ScanParams &p, const BlockCtx &c, uint32_t row) {
  uint32_t stack = 0;
  for (int i = 0; i < p.n_nodes; ++i) {
    const FilterNodeDev &nd = p.nodes[i];
    bool r;
    if (nd.kind == NODE_WHITE) {
      r = eval_leaf(p, c, nd, row);
    } else {
      const uint32_t m = (1u << nd.n_children) - 1u;
      const uint32_t top = stack & m;
      r = nd.kind == NODE_AND ? top == m : top != 0;
      stack >>= nd.n_children;
    }
    stack = (stack << 1) | (r ? 1u : 0u);
  }
  return stack & 1u;
}

// Number of leading dictionary indexes for which `pred` holds (pred is monotone over a sorted dictionary: true ...
// true false ... false). Warp-cooperative 32-ary search: every round probes 32 evenly spaced entries, so a
// 1 K-entry dictionary takes two rounds (the reference binary-searches, std::lower_bound / upper_bound over
// ObDictDecoderIterator, encoding/ob_dict_decoder.cpp:967-988,1085-1176).
template <typename Pred>
__device__ __forceinline__ uint32_t warp_partition_point(uint32_t n, int lane, Pred pred) {
  uint32_t lo = 0, hi = n;
  while (lo < hi) {
    const uint32_t step = (hi - lo + 31u) >> 5;
    const uint32_t idx = lo + (uint32_t)lane * step;
    const uint32_t k = __popc(__ballot_sync(0xffffffffu, idx < hi && pred(idx)));  // true probes form a prefix
    if (k == 0) break;
    const uint32_t last_true = lo + (k - 1u) * step;
    lo = last_true + 1u;
    hi = min(hi, last_true + step);
  }
  return lo;
}

__device__ __forceinline__ uint32_t range_word(uint32_t a, uint32_t b, uint32_t w) {   // bits of [a, b) that fall in word w
  const uint32_t lo = w * 32u, s = a > lo ? a : lo, e = b < lo + 32u ? b : lo + 32u;
  if (s >= e) return 0u;
  const uint32_t len = e - s;
  return (len == 32u ? 0xffffffffu : ((1u << len) - 1u)) << (s - lo);
}

// Sorted fixed-length dictionary (IS_SORTED): the matching refs of a comparison form one index interval [a, b),
// found by searching the constants instead of evaluating every entry (fast_cmp_ref_and_set_res,
// ob_dict_decoder.cpp:1426). Returns false when the leaf does not have that shape (IN lists, NU / NN, ...).
__device__ __forceinline__ bool build_dict_bitset_sorted(const ScanParams &p, const BlockView &b, const ColDesc &d,
                                                         const FilterNodeDev &nd, uint32_t *bits, const Team &t) {
  const uint32_t n = d.dict_count;
  const int op = nd.op;
  uint32_t a = 0, e = 0;
  bool neg = false;
  if (d.sc != 5) {
    if (!nd.range_ok) return false;
    const bool sg = d.sc == 1;
    const uint64_t lo = nd.lo, hi = nd.lo + nd.span;
    auto lt = [&](uint64_t x, uint64_t y) { return sg ? (int64_t)x < (int64_t)y : x < y; };
    a = warp_partition_point(n, t.lane, [&](uint32_t i) { return lt((uint64_t)cmp_image(d, dict_int(b.s, d, i)), lo); });
    e = warp_partition_point(n, t.lane, [&](uint32_t i) { return !lt(hi, (uint64_t)cmp_image(d, dict_int(b.s, d, i))); });
    neg = nd.negate != 0;
  } else {
    if (op > OP_BT) return false;
    const uint32_t len = d.dict_data_size;
    auto cmpk = [&](uint32_t i, int k) {
      const ParamDev &pp = p.params[nd.param_begin + k];
      return str_cmp(b.s, d.dict_payload + i * len, len, p.param_heap + pp.heap_off, pp.len);
    };
    const int k_hi = op == OP_BT ? 1 : 0;
    const bool need_lb = op == OP_EQ || op == OP_NE || op == OP_GE || op == OP_BT || op == OP_LT;
    const bool need_ub = op == OP_EQ || op == OP_NE || op == OP_LE || op == OP_BT || op == OP_GT;
    uint32_t lb = 0, ub = 0;
    if (need_lb) lb = warp_partition_point(n, t.lane, [&](uint32_t i) { return cmpk(i, 0) < 0; });       // first entry >= c0
    if (need_ub) ub = warp_partition_point(n, t.lane, [&](uint32_t i) { return cmpk(i, k_hi) <= 0; });   // first entry > c (c1 for BT)
    switch (op) {
      case OP_EQ: a = lb; e = ub; break;
      case OP_NE: a = lb; e = ub; neg = true; break;
      case OP_LT: a = 0; e = lb; break;
      case OP_LE: a = 0; e = ub; break;
      case OP_GE: a = lb; e = n; break;
      case OP_GT: a = ub; e = n; break;
      default: a = lb; e = ub; break;   // BT
    }
  }
  if (e < a) e = a;
  const uint32_t nw = (n + 2u + 31u) >> 5;
  for (uint32_t w = (uint32_t)t.warp * 32u + (uint32_t)t.lane; w < nw; w += (uint32_t)t.nwarps * 32u) {
    uint32_t m = range_word(a, e, w);
    if (neg) m = ~m & range_word(0, n, w);   // NE: every non-NULL ref outside the interval
    bits[w] = m;                             // refs n (NULL) and n + 1 (NOP) never match a comparison
  }
  return true;
}

// Predicate over the dictionary of a DICT / RLE column -> bitset over refs (bit count = NULL ref).
__device__ __forceinline__ void build_dict_bitset(const ScanParams &p, const BlockView &b, const ColDesc &d,
                                                  const FilterNodeDev &nd, uint32_t *bits, const Team &t) {
  const uint32_t n = d.dict_count + 2;
  const int op = nd.op;
  if (d.dict_sorted && t.nwarps == 1 && op != OP_FALSE && op != OP_TRUE && build_dict_bitset_sorted(p, b, d, nd, bits, t)) return;
  for (uint32_t base = (uint32_t)t.warp * 32u; base < n; base += (uint32_t)t.nwarps * 32u) {
    const uint32_t idx = base + (uint32_t)t.lane;
    bool r = false;
    if (idx < d.dict_count) {
      if (op == OP_NN) r = true;
      else if (op == OP_NU) r = false;
      else if (d.sc == 5) {
        uint32_t cell, len;
        dict_str(b.s, d, idx, cell, len);
        r = str_pred(p, nd, b.s, cell, len);
      } else {
        r = int_pred(p, nd, d, dict_int(b.s, d, idx));
      }
    } else if (idx == d.dict_count) {
      r = op == OP_NU;
    }
    const uint32_t word = __ballot_sync(0xffffffffu, r);
    if (t.lane == 0) bits[base >> 5] = word;
  }
}

__device__ __forceinline__ uint32_t valid_mask_of(uint32_t rows, uint32_t g) {
  const uint32_t rem = rows - g * 32u;
  return rem >= 32u ? 0xffffffffu : ((1u << rem) - 1u);
}

// Range test over a K_BITS column without NULLs / sign fix: the hot filter loop.
//   MODE 0: first leaf (bm[g] = leaf), 1: AND into bm with early-out, 2: OR into bm with early-out
//   G: the block is read straight from global memory (count kernel) instead of shared memory
//   NARROW: datum narrower than 8 bytes (date, year, ...): the compare image is the low elem_len bytes of
//   value + base, sign-extended for signed classes (cmp_image) -- done with and / xor / sub on the lane
template <bool WIDE, int MODE, bool G, bool NARROW>
__device__ __forceinline__ void filter_bits_range(const BlockCtx &c, const ColDesc &d, const FilterNodeDev &nd,
                                                  uint32_t *bm, uint32_t rows, uint32_t nwords, const Team &t) {
  const uint32_t stride = d.stride, width = d.width;
  const uint64_t lo = NARROW ? nd.lo : nd.lo - d.base, span = nd.span;  // (v + base - lo) <= span
  const uint64_t nbase = d.base, nmask = d.elem_len == 4 ? 0xffffffffull : 0xffull;
  const uint64_t nsign = (d.elem_len == 4 && d.sc == 1) ? 0x80000000ull : 0ull;
  const bool neg = nd.negate != 0;
  const uint32_t nfull = rows >> 5;
  const uint32_t step = (uint32_t)t.nwarps * 32u * stride;
  const uint8_t *gs = c.b.s;
  uint32_t bit = (G ? 0u : c.sbit) + d.val_bit + ((uint32_t)t.warp * 32u + (uint32_t)t.lane) * stride;
  uint32_t g = (uint32_t)t.warp;
  auto load = [&](uint32_t bo) -> uint64_t {
    uint64_t v;
    if (G) v = WIDE ? ld_bits(gs, bo, width) : (uint64_t)ld_bits32(gs, bo, width);
    else v = WIDE ? sbits(bo, width) : (uint64_t)sbits32(bo, width);
    if (NARROW) v = ((((v + nbase) & nmask) ^ nsign) - nsign);
    return v;
  };
  for (; g < nfull; g += (uint32_t)t.nwarps, bit += step) {
    uint32_t cur = 0;
    if (MODE != 0) {
      cur = bm[g];
      if (MODE == 1 ? cur == 0u : cur == 0xffffffffu) continue;
    }
    const uint64_t v = load(bit);
    const uint32_t w = __ballot_sync(0xffffffffu, ((v - lo) <= span) != neg);
    if (t.lane == 0) bm[g] = MODE == 0 ? w : (MODE == 1 ? (cur & w) : (cur | w));
  }
  if (g < nwords) {  // ragged tail group: lanes past the last row must not touch memory
    const uint32_t vm = valid_mask_of(rows, g);
    const uint32_t cur = MODE == 0 ? 0u : bm[g];
    const uint64_t v = g * 32u + (uint32_t)t.lane < rows ? load(bit) : 0ull;
    const uint32_t w = __ballot_sync(0xffffffffu, ((v - lo) <= span) != neg) & vm;
    if (t.lane == 0) bm[g] = MODE == 0 ? w : (MODE == 1 ? (cur & w) : (cur | w));
  }
}

__device__ __forceinline__ bool leaf_is_bits_range(const ColDesc &d, const FilterNodeDev &nd) {
  return d.kind == K_BITS && nd.range_ok && d.ext_bit == 0 && !d.sign_fix && !d.var_is_last;
}


// ---- byte-aligned columns: one LANE per 32 rows, SIMD-in-register compares ----------------------------
// For value arrays of whole bytes (every CS integer stream, PAX byte-packed columns) a lane owns a whole
// bitmap word: it reads its 32 values as 32-bit words from the staged column (funnel-shifted to the value
// alignment), tests 4 (or 2) values per instruction with the per-byte (halfword) video instructions and
// packs the compare masks into its own bitmap word. No ballot, ~50 warp instructions per 1024 rows.
// The range lo..hi is first moved into the raw (value - base) domain with 128-bit arithmetic.
struct RawRange { uint32_t lo, span; bool none; };
__device__ __forceinline__ RawRange raw_range_of(const ColDesc &d, const FilterNodeDev &nd, uint32_t bytes) {
  const bool sg = d.sc == 1;
  const uint64_t hi64 = nd.lo + nd.span;
  const __int128 lo = sg ? (__int128)(int64_t)nd.lo : (__int128)nd.lo;
  const __int128 hi = sg ? (__int128)(int64_t)hi64 : (__int128)hi64;
  const __int128 base = sg ? (__int128)(int64_t)d.base : (__int128)d.base;
  const __int128 vmax = ((__int128)1 << (bytes * 8u)) - 1;
  __int128 l = lo - base, h = hi - base;
  RawRange r;
  r.none = h < 0 || l > vmax || l > h;
  if (l < 0) l = 0;
  if (h > vmax) h = vmax;
  r.lo = (uint32_t)l;
  r.span = r.none ? 0u : (uint32_t)(h - l);
  return r;
}
// may the raw-domain test stand in for the compare image of this column? (narrow signed datums: only when
// base + raw cannot leave the datum's range, which valid data never does)
__device__ __forceinline__ bool simd_domain_ok(const ColDesc &d, uint32_t bytes) {
  if (d.elem_len == 8) return true;
  if (d.elem_len == 4 && d.sc == 1) {
    const int64_t b = (int64_t)d.base, top = b + (int64_t)((1ull << (bytes * 8u)) - 1ull);
    return b >= (int64_t)INT32_MIN && top <= (int64_t)INT32_MAX;
  }
  return false;
}
__device__ __forceinline__ bool leaf_is_bytes_simd(const ColDesc &d, const FilterNodeDev &nd) {
  return d.kind == K_BITS && nd.range_ok && d.ext_bit == 0 && !d.sign_fix && !d.var_is_last && d.stride == d.width &&
         (d.width == 8 || d.width == 16) && (d.val_bit & 7u) == 0 && simd_domain_ok(d, d.width >> 3);
}
template <int BYTES, int MODE>
__device__ __forceinline__ void filter_bytes_simd(const BlockCtx &c, const ColDesc &d, const FilterNodeDev &nd, uint32_t *bm,
                                                  uint32_t rows, uint32_t nwords, const Team &t) {
  const RawRange rr = raw_range_of(d, nd, BYTES);
  const bool neg = nd.negate != 0;
  const uint32_t lo4 = BYTES == 1 ? rr.lo * 0x01010101u : rr.lo * 0x00010001u;
  const uint32_t sp4 = BYTES == 1 ? rr.span * 0x01010101u : rr.span * 0x00010001u;
  const uint32_t vbyte = (c.sbit + d.val_bit) >> 3;  // shared-window byte address of value 0
  constexpr uint32_t kWordsPerGroup = 8u * BYTES;     // 32-bit words holding 32 values
  for (uint32_t g = (uint32_t)t.tid; g < nwords; g += (uint32_t)t.nthreads) {
    uint32_t cur = 0;
    if (MODE != 0) {
      cur = bm[g];
      if (MODE == 1 ? cur == 0u : cur == 0xffffffffu) continue;
    }
    const uint32_t vm = valid_mask_of(rows, g);
    uint32_t m = 0;
    if (!rr.none) {
      const uint32_t nvalid = rows - g * 32u < 32u ? rows - g * 32u : 32u;
      const uint32_t kmax = (nvalid * BYTES + 3u) >> 2;  // words that hold valid rows: never read past the column
      const uint32_t first = vbyte + g * 32u * BYTES;
      const uint32_t a = first & ~3u, sh = (first & 3u) * 8u;
      uint32_t w0 = sld32(a);
#pragma unroll
      for (uint32_t k = 0; k < kWordsPerGroup; ++k) {
        if (k < kmax) {
          const uint32_t w1 = sld32(a + 4u * k + 4u);
          const uint32_t v = __funnelshift_r(w0, w1, sh);
          w0 = w1;
          if (BYTES == 1) {
            const uint32_t hit = __vcmpleu4(__vsub4(v, lo4), sp4) & 0x01010101u;
            m |= (((hit * 0x01020408u) >> 24) & 0xfu) << (4u * k);
          } else {
            const uint32_t hit = __vcmpleu2(__vsub2(v, lo4), sp4) & 0x00010001u;
            m |= ((hit | (hit >> 15)) & 0x3u) << (2u * k);
          }
        }
      }
    }
    if (neg) m = ~m;
    m &= vm;
    bm[g] = MODE == 0 ? m : (MODE == 1 ? (cur & m) : (cur | m));
  }
}

// First leaf of an AND / OR list: writes bm directly (no initialisation pass) when it is a plain
// range test. Returns false if the caller has to initialise bm and run the leaf generically.
template <bool G>
__device__ __forceinline__ bool leaf_first_fast(const ScanParams &p, const BlockCtx &c, const FilterNodeDev &nd,
                                                uint32_t *bm, uint32_t rows, uint32_t nwords, const Team &t) {
  if (nd.kind != NODE_WHITE) return false;
  const ColDesc &d = c.descs[nd.used_idx];
  if (!leaf_is_bits_range(d, nd)) return false;
  if (!G && leaf_is_bytes_simd(d, nd)) {
    if (d.width == 8) filter_bytes_simd<1, 0>(c, d, nd, bm, rows, nwords, t);
    else filter_bytes_simd<2, 0>(c, d, nd, bm, rows, nwords, t);
    return true;
  }
  if (d.elem_len != 8) {
    if (d.width <= 32) filter_bits_range<false, 0, G, true>(c, d, nd, bm, rows, nwords, t);
    else filter_bits_range<true, 0, G, true>(c, d, nd, bm, rows, nwords, t);
  } else if (d.width <= 32) filter_bits_range<false, 0, G, false>(c, d, nd, bm, rows, nwords, t);
  else filter_bits_range<true, 0, G, false>(c, d, nd, bm, rows, nwords, t);
  return true;
}

// One leaf evaluated column-at-a-time over the ballot words owned by this warp (g = warp, warp+n,
// ...). `and_mode`: bm[g] &= leaf, skipping groups that are already all-false; else bm[g] |= leaf
// for groups that are not yet all-true (the reference's can_skip_filter / early-out, per 32 rows).
template <bool G>
__device__ __forceinline__ void leaf_over_words(const ScanParams &p, const BlockCtx &c, const FilterNodeDev &nd,
                                                uint32_t *bm, uint32_t rows, uint32_t nwords, bool and_mode,
                                                const Team &t) {
  const ColDesc &d = c.descs[nd.used_idx];
  const int op = nd.op;
  // ---- fast path A: integer range test on a K_BITS column without NULLs ------------------------------
  if (leaf_is_bits_range(d, nd)) {
    if (!G && leaf_is_bytes_simd(d, nd)) {
      if (d.width == 8) {
        if (and_mode) filter_bytes_simd<1, 1>(c, d, nd, bm, rows, nwords, t);
        else filter_bytes_simd<1, 2>(c, d, nd, bm, rows, nwords, t);
      } else {
        if (and_mode) filter_bytes_simd<2, 1>(c, d, nd, bm, rows, nwords, t);
        else filter_bytes_simd<2, 2>(c, d, nd, bm, rows, nwords, t);
      }
      return;
    }
    if (d.elem_len != 8) {
      if (d.width <= 32) {
        if (and_mode) filter_bits_range<false, 1, G, true>(c, d, nd, bm, rows, nwords, t);
        else filter_bits_range<false, 2, G, true>(c, d, nd, bm, rows, nwords, t);
      } else {
        if (and_mode) filter_bits_range<true, 1, G, true>(c, d, nd, bm, rows, nwords, t);
        else filter_bits_range<true, 2, G, true>(c, d, nd, bm, rows, nwords, t);
      }
    } else if (d.width <= 32) {
      if (and_mode) filter_bits_range<false, 1, G, false>(c, d, nd, bm, rows, nwords, t);
      else filter_bits_range<false, 2, G, false>(c, d, nd, bm, rows, nwords, t);
    } else {
      if (and_mode) filter_bits_range<true, 1, G, false>(c, d, nd, bm, rows, nwords, t);
      else filter_bits_range<true, 2, G, false>(c, d, nd, bm, rows, nwords, t);
    }
    return;
  }
  // ---- fast path B: DICT column through the predicate bitset ------------------------------------------
  if (d.kind == K_DICT && op != OP_FALSE && op != OP_TRUE) {
    const uint32_t *bits = c.bitsets + nd.slot * p.bitset_words;
    const uint32_t cntp1 = d.dict_count + 1;
    const uint32_t val_bit = (G ? 0u : c.sbit) + d.val_bit, stride = d.stride, width = d.width;
    const uint8_t *gs = c.b.s;
    const uint32_t nfull = rows >> 5;
    uint32_t g = (uint32_t)t.warp;
    uint32_t bit = val_bit + ((uint32_t)t.warp * 32u + (uint32_t)t.lane) * stride;
    const uint32_t step = (uint32_t)t.nwarps * 32u * stride;
    for (; g < nfull; g += (uint32_t)t.nwarps, bit += step) {  // full words: no row bound, no valid mask
      const uint32_t cur = bm[g];
      if (and_mode ? cur == 0u : cur == 0xffffffffu) continue;
      uint32_t ref = G ? ld_bits32(gs, bit, width) : sbits32(bit, width);
      ref = ref < cntp1 ? ref : cntp1;
      const uint32_t w = __ballot_sync(0xffffffffu, (bits[ref >> 5] >> (ref & 31)) & 1u);
      if (t.lane == 0) bm[g] = and_mode ? (cur & w) : (cur | w);
    }
    if (g < nwords) {  // ragged tail: lanes past the last row must not touch memory
      const uint32_t cur = bm[g], vm = valid_mask_of(rows, g);
      if (!(and_mode ? cur == 0u : cur == vm)) {
        uint32_t ref = cntp1;
        if (g * 32u + (uint32_t)t.lane < rows) ref = G ? ld_bits32(gs, bit, width) : sbits32(bit, width);
        ref = ref < cntp1 ? ref : cntp1;
        const uint32_t w = __ballot_sync(0xffffffffu, (bits[ref >> 5] >> (ref & 31)) & 1u) & vm;
        if (t.lane == 0) bm[g] = and_mode ? (cur & w) : (cur | w);
      }
    }
    return;
  }
  // ---- generic leaf (RLE via the predicate bitset + run lookup, strings, NULL-able columns, ...) ----
  for (uint32_t g = (uint32_t)t.warp; g < nwords; g += (uint32_t)t.nwarps) {
    const uint32_t cur = bm[g], vm = valid_mask_of(rows, g);
    if (and_mode ? cur == 0u : cur == vm) continue;
    const uint32_t row = g * 32u + (uint32_t)t.lane;
    const bool pr = row < rows && eval_leaf(p, c, nd, row);
    const uint32_t w = __ballot_sync(0xffffffffu, pr) & vm;
    if (t.lane == 0) bm[g] = and_mode ? (cur & w) : (cur | w);
  }
}

// =================================================================================================
// Block-wide helpers
// =================================================================================================
// Loads a block into shared memory with one TMA bulk transaction; all threads return once the
// bytes have landed. `bar` must have been initialised by thread 0 (count 1) before the call.
__device__ __forceinline__ void load_block(uint8_t *smem, const uint8_t *src, uint32_t bytes16, uint64_t *bar,
                                           uint32_t parity) {
  if (threadIdx.x == 0) {
    mbar_expect_tx(bar, bytes16);
    tma_bulk_g2s(smem, src, bytes16, bar);
  }
  mbar_wait(bar, parity);
}

// Builds the run table of RLE column d (see RleTable) with the whole team.
__device__ __forceinline__ void rle_table_build(const uint8_t *s, const ColDesc &d, uint32_t rows, uint32_t *mask,
                                                uint16_t *pre, const Team &t) {
  const uint32_t nwords = (rows + 31u) >> 5;
  for (uint32_t g = (uint32_t)t.tid; g < nwords; g += (uint32_t)t.nthreads) mask[g] = 0u;
  t.sync();
  for (uint32_t k = (uint32_t)t.tid; k < d.rle_count; k += (uint32_t)t.nthreads) {
    const uint32_t start = ld_bits32(s, d.rle_row_ids_bit + k * d.rle_row_id_bits, d.rle_row_id_bits);
    if (start < rows) atomicOr(&mask[start >> 5], 1u << (start & 31u));
  }
  t.sync();
  if (t.tid < 32) {
    uint32_t carry = 0;
    for (uint32_t base = 0; base < nwords; base += 32u) {
      const uint32_t g = base + (uint32_t)t.tid;
      const uint32_t c = g < nwords ? (uint32_t)__popc(mask[g]) : 0u;
      uint32_t inc = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
        if ((t.tid & 31) >= o) inc += u;
      }
      if (g < nwords) pre[g] = (uint16_t)(carry + inc - c);
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
  }
  t.sync();
}

// Parses the staged block (at g_smem + soff) and builds descriptors + RLE run tables. Returns false
// (uniformly over the team) when the block cannot be handled; *corrupt tells why.
__device__ __forceinline__ bool prepare_block(const ScanParams &p, uint32_t soff, uint32_t size, ColDesc *descs,
                                              uint8_t *rle_base, const Team &t, BlockCtx &c, bool &corrupt) {
  const uint8_t *sblk = g_smem + soff;
  // every thread parses the 64-byte header itself (a handful of shared-memory loads): no barrier
  parse_block(sblk, size, c.b);
  if (c.b.ok && c.b.row_count > p.rows_cap) c.b.ok = 0;
  c.sbit = (smem_u32(g_smem) + soff) * 8u;
  corrupt = !c.b.ok;
  bool my_bad = false;
  // descriptors are built by the last threads of the team
  const int di = t.nthreads - 1 - t.tid;
  if (c.b.ok && di < p.n_used) {
    ColDesc d;
    build_col_desc(c.b, p.used_col[di], d);
    d.rle_slot = d.kind == K_RLE ? p.used_rle_slot[di] : (int8_t)-1;
    if (d.kind == K_RLE && d.rle_slot >= 0 && d.rle_count > (uint32_t)p.rle_runs_cap) d.ok = 0;
    descs[di] = d;
    my_bad = !d.ok;
  }
  const bool bad = t.sync_or(my_bad || !c.b.ok);
  c.descs = descs;
  c.rle_base = rle_base;
  c.rle_slot_bytes = p.rle_slot_bytes;
  c.rle_starts_bytes = p.words_cap * 4u;
  if (bad) return false;
  // RLE run tables
  if (p.n_rle_slots > 0) {
    for (int i = 0; i < p.n_used; ++i) {
      if (p.used_rle_slot[i] < 0) continue;
      const ColDesc &d = descs[i];
      if (d.kind != K_RLE) continue;
      uint8_t *slot = rle_base + (uint32_t)d.rle_slot * p.rle_slot_bytes;
      rle_table_build(sblk, d, c.b.row_count, reinterpret_cast<uint32_t *>(slot),
                      reinterpret_cast<uint16_t *>(slot + c.rle_starts_bytes), t);
    }
  }
  return true;
}

// =================================================================================================
// Projection of one column over the selected rows (column-at-a-time, specialised)
// =================================================================================================
// Output vectors are written once and never read again by the scan: streaming stores (st.global.cs) keep them from
// evicting the block bytes the count kernel has just pulled through L2.
#define ROW(j) (IDENT ? (uint32_t)(j) : (uint32_t)sel[j])
template <typename OutT, bool IDENT>
__device__ __forceinline__ void project_int_col(const ScanParams &p, const BlockCtx &c, const ColDesc &d, int pc,
                                                const uint16_t *sel, uint32_t cnt, int64_t base_row, const Team &t) {
  OutT *out = reinterpret_cast<OutT *>(p.out_data[pc]) + base_row;
  const uint32_t tid = (uint32_t)t.tid, nt = (uint32_t)t.nthreads;
  bool saw_null = false;
  auto mark_null = [&](uint32_t j) {
    const int64_t o = base_row + (int64_t)j;
    atomicOr(&p.out_nulls[pc][o >> 5], 1u << (o & 31));
    saw_null = true;
  };
  if (d.kind == K_BITS) {
    const uint32_t val_bit = c.sbit + d.val_bit, stride = d.stride, width = d.width;
    const uint64_t add = d.base, mask = d.int_mask;
    const bool fix = d.sign_fix != 0;
    if (d.ext_bit == 0 && !fix && !d.var_is_last) {
      if (width <= 32) {
        for (uint32_t j = tid; j < cnt; j += nt)
          __stcs(&out[j], (OutT)((uint64_t)sbits32(val_bit + ROW(j) * stride, width) + add));
      } else {
        for (uint32_t j = tid; j < cnt; j += nt)
          __stcs(&out[j], (OutT)(sbits(val_bit + ROW(j) * stride, width) + add));
      }
    } else {
      const uint32_t ext_off = c.sbit + d.ext_bit_off, eb = d.ext_bit, exor = d.var_ext_in_row;
      const bool repl = d.var_is_last != 0;
      const uint64_t repl_raw = null_replaced_raw(d);
      for (uint32_t j = tid; j < cnt; j += nt) {
        const uint32_t row = ROW(j);
        if (eb && sbits32(ext_off + (row ^ exor) * eb, eb) != STORED_NOT_EXT) {
          __stcs(&out[j], (OutT)0);
          mark_null(j);
          continue;
        }
        const uint64_t raw = sbits(val_bit + row * stride, width);
        if (repl && raw == repl_raw) {
          __stcs(&out[j], (OutT)0);
          mark_null(j);
          continue;
        }
        uint64_t v = raw + add;
        if (fix) v = sign_fix(mask, v);
        __stcs(&out[j], (OutT)v);
      }
    }
  } else {  // K_DICT / K_RLE
    const uint32_t dcount = d.dict_count, dbits = d.dict_data_size * 8u, dpay = c.sbit + d.dict_payload * 8u;
    const uint64_t mask = d.int_mask, dbase = d.base;
    const bool fix = d.sign_fix != 0;
    if (d.kind == K_DICT) {
      const uint32_t val_bit = c.sbit + d.val_bit, stride = d.stride, width = d.width;
      for (uint32_t j = tid; j < cnt; j += nt) {
        const uint32_t ref = sbits32(val_bit + ROW(j) * stride, width);
        if (ref >= dcount) {
          __stcs(&out[j], (OutT)0);
          mark_null(j);
          continue;
        }
        uint64_t v = sbits(dpay + ref * dbits, dbits) + dbase;
        if (fix) v = sign_fix(mask, v);
        __stcs(&out[j], (OutT)v);
      }
    } else if (d.rle_slot >= 0) {
      const RleTable rt = c.rle_table(d.rle_slot);
      const uint32_t refs_bit = c.sbit + d.rle_refs_bit, ref_bits = d.rle_ref_bits;
      for (uint32_t j = tid; j < cnt; j += nt) {
        const uint32_t ref = sbits32(refs_bit + rle_run_of(rt, ROW(j)) * ref_bits, ref_bits);
        if (ref >= dcount) {
          __stcs(&out[j], (OutT)0);
          mark_null(j);
          continue;
        }
        uint64_t v = sbits(dpay + ref * dbits, dbits);
        if (fix) v = sign_fix(mask, v);
        __stcs(&out[j], (OutT)v);
      }
    } else {
      for (uint32_t j = tid; j < cnt; j += nt) {
        bool is_null;
        const uint64_t v = int_cell(c.b, d, nullptr, ROW(j), is_null);
        __stcs(&out[j], (OutT)(is_null ? 0ull : v));
        if (is_null) mark_null(j);
      }
    }
  }
  if (saw_null) p.has_null[pc] = 1;
}

// Same projection through generic loads on the block in global memory (sparse selections).
template <typename OutT>
__device__ __forceinline__ void project_int_col_global(const ScanParams &p, const BlockCtx &c, const ColDesc &d, int pc,
                                                       const uint16_t *sel, uint32_t cnt, int64_t base_row, const Team &t) {
  OutT *out = reinterpret_cast<OutT *>(p.out_data[pc]) + base_row;
  bool saw_null = false;
  for (uint32_t j = (uint32_t)t.tid; j < cnt; j += (uint32_t)t.nthreads) {
    bool is_null;
    const uint64_t v = int_cell(c.b, d, nullptr, (uint32_t)sel[j], is_null);
    __stcs(&out[j], (OutT)(is_null ? 0ull : v));
    if (is_null) {
      const int64_t o = base_row + (int64_t)j;
      atomicOr(&p.out_nulls[pc][o >> 5], 1u << (o & 31));
      saw_null = true;
    }
  }
  if (saw_null) p.has_null[pc] = 1;
}

template <bool IDENT>
__device__ __forceinline__ void project_str_col(const ScanParams &p, const BlockCtx &c, const ColDesc &d, int pc,
                                                const uint16_t *sel, uint32_t cnt, int64_t base_row,
                                                uint64_t blk_addr, const Team &t) {
  uint64_t *optr = reinterpret_cast<uint64_t *>(p.out_data[pc]) + base_row;
  int32_t *olen = p.out_lens[pc] + base_row;
  RleTable rt{};
  const RleTable *rtp = nullptr;
  if (d.kind == K_RLE && d.rle_slot >= 0) {
    rt = c.rle_table(d.rle_slot);
    rtp = &rt;
  }
  bool saw_null = false;
  for (uint32_t j = (uint32_t)t.tid; j < cnt; j += (uint32_t)t.nthreads) {
    uint32_t cell, len;
    bool is_null;
    str_cell(c.b, d, rtp, ROW(j), cell, len, is_null);
    __stcs(&optr[j], is_null ? 0ull : blk_addr + cell);
    __stcs(&olen[j], is_null ? 0 : (int32_t)len);
    if (is_null) {
      const int64_t o = base_row + (int64_t)j;
      atomicOr(&p.out_nulls[pc][o >> 5], 1u << (o & 31));
      saw_null = true;
    }
  }
  if (saw_null) p.has_null[pc] = 1;
}

#undef ROW

// One projected column of one block decoded by ONE WARP from the staged image (c.b.s / c.sbit already point at the
// column's staged bytes): RLE columns get their run table (and, for 8-byte integers, their run values) in the warp's
// private scratch `wscr` first. Shared by the CTA-per-block and the warp-per-block projection kernels.
__device__ __forceinline__ void project_column_staged(const ScanParams &p, BlockCtx &c, ColDesc *wdesc, int pc, const uint16_t *sel,
                                                      uint32_t cnt, int64_t base, uint64_t blk_addr, bool all_rows, uint32_t rows,
                                                      uint8_t *wscr, const Team &t) {
  const int lane = t.lane;
  const ColDesc &d = *wdesc;
  if (!d.ok) {
    if (lane == 0) atomicOr(p.status, ST_UNSUPPORTED);
    return;
  }
  if (d.kind == K_RLE) {
    if (d.rle_count > (uint32_t)p.rle_runs_cap) {
      if (lane == 0) atomicOr(p.status, ST_UNSUPPORTED);
      return;
    }
    if (lane == 0) wdesc->rle_slot = 0;
    rle_table_build(c.b.s, d, rows, reinterpret_cast<uint32_t *>(wscr + p.pw_rle),
                    reinterpret_cast<uint16_t *>(wscr + p.pw_rle + c.rle_starts_bytes), t);
    const uint32_t n = d.rle_count;
    if (d.sc != 5 && d.elem_len == 8) {
      // integer RLE column: decode each RUN once (value of run k), rows then only look up their run
      uint64_t *rvals = reinterpret_cast<uint64_t *>(wscr + p.pw_rvals);
      const uint32_t refs_bit = c.sbit + d.rle_refs_bit, ref_bits = d.rle_ref_bits;
      const uint32_t dcount = d.dict_count, dbits = d.dict_data_size * 8u, dpay = c.sbit + d.dict_payload * 8u;
      bool null_run = false;
      for (uint32_t k = (uint32_t)lane; k < n; k += 32u) {
        const uint32_t ref = sbits32(refs_bit + k * ref_bits, ref_bits);
        uint64_t v = 0;
        if (ref >= dcount) null_run = true;
        else {
          v = sbits(dpay + ref * dbits, dbits);
          if (d.sign_fix) v = sign_fix(d.int_mask, v);
        }
        rvals[k] = v;
      }
      const bool any_null = __any_sync(0xffffffffu, null_run);
      __syncwarp();
      if (!any_null) {
        uint64_t *out = reinterpret_cast<uint64_t *>(p.out_data[pc]) + base;
        const RleTable rt = c.rle_table(0);
        if (all_rows) for (uint32_t j = (uint32_t)lane; j < cnt; j += 32u) __stcs(&out[j], rvals[rle_run_of(rt, j)]);
        else for (uint32_t j = (uint32_t)lane; j < cnt; j += 32u) __stcs(&out[j], rvals[rle_run_of(rt, sel[j])]);
        return;
      }
    }
  }
  if (all_rows) {
    if (d.sc == 5) project_str_col<true>(p, c, d, pc, sel, cnt, base, blk_addr, t);
    else if (d.elem_len == 8) project_int_col<uint64_t, true>(p, c, d, pc, sel, cnt, base, t);
    else if (d.elem_len == 4) project_int_col<uint32_t, true>(p, c, d, pc, sel, cnt, base, t);
    else project_int_col<uint8_t, true>(p, c, d, pc, sel, cnt, base, t);
  } else {
    if (d.sc == 5) project_str_col<false>(p, c, d, pc, sel, cnt, base, blk_addr, t);
    else if (d.elem_len == 8) project_int_col<uint64_t, false>(p, c, d, pc, sel, cnt, base, t);
    else if (d.elem_len == 4) project_int_col<uint32_t, false>(p, c, d, pc, sel, cnt, base, t);
    else project_int_col<uint8_t, false>(p, c, d, pc, sel, cnt, base, t);
  }
}

// =================================================================================================
// Index kernel (batch open): one thread per (block, column) parses the block straight from HBM and
// stores the column's decode plan. The scan kernels never parse headers; the reference keeps the
// same kind of cached decoder state beside a block in its block cache (ObBlockCachedDecoderHeader,
// blocksstable/ob_micro_block_cache.cpp:1345-1363).
// =================================================================================================
__global__ void __launch_bounds__(256) obgpu_index_kernel(const uint8_t *image, const uint64_t *blk_off,
                                                          const uint32_t *blk_size, const int64_t *bm_word_off,
                                                          int n_blocks, int max_cols, ColDesc *plans, uint32_t *rows,
                                                          BlockRec *recs, uint32_t *col_span) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)n_blocks * max_cols) return;
  const int block = (int)(i / max_cols), col = (int)(i % max_cols);
  BlockView b;
  parse_block(image + blk_off[block], blk_size[block], b);
  ColDesc d{};
  d.rle_slot = -1;
  if (b.ok) build_col_desc(b, col, d);
  plans[i] = d;
  if (col == 0) {
    rows[block] = b.ok ? b.row_count : 0u;
    BlockRec r{};
    r.off = blk_off[block];
    r.bm_word_off = bm_word_off[block];
    r.size = blk_size[block];
    r.rows = b.ok ? b.row_count : 0u;
    r.row_data_off = b.row_data_off;
    r.row_index_off = b.row_index_off;
    r.header_size = b.header_size;
    r.column_count = (uint16_t)b.column_count;
    r.var_col_cnt = b.var_col_cnt;
    r.row_index_byte = b.row_index_byte;
    r.ext_bit = b.ext_bit;
    r.pad[0] = b.is_cs;
    recs[block] = r;
  }
  if (d.ok) {
    // bytes of the column's region (count kernel staging buffer, project kernel column staging)
    uint32_t lo, hi;
    if (col_region(d, b, lo, hi)) atomicMax(&col_span[col], hi - lo);
    else atomicMax(&col_span[col], 0xffffffffu);   // no single region (CS string bytes): whole-block staging only
    // dictionary size (predicate bitset words) of dictionary-coded columns: col_span[max_cols + col]
    if (is_dict_kind(d)) atomicMax(&col_span[max_cols + col], d.dict_count + 2u);
    // bytes a projection of the column stages (scan_small.cuh: VARCHAR dictionaries without their string bytes)
    atomicMax(&col_span[5 * max_cols + col], proj_ranges_bytes(d, b));
    // strings that exist only in this batch's copy of the block (HEX_PACKING / STRING_DIFF / STRING_PREFIX, mat_codecs.cuh)
    if (d.kind == K_CSSTR && !b.is_cs) atomicMax(&col_span[6 * max_cols + col], 1u);
  }
  if (b.ok && (uint32_t)col < b.column_count) {
    // per-column facts the host keeps for a batch: ObObjType (min / max over the blocks: equal when the blocks
    // agree) and the largest RLE run count (sizes the run tables)
    const uint8_t *s = image + blk_off[block];
    const uint32_t t = b.is_cs ? s[b.header_size + 12u + 4u * (uint32_t)col + 3u] : s[b.header_size + 16u * (uint32_t)col + 3u];
    atomicMin(&col_span[2 * max_cols + col], t);
    atomicMax(&col_span[3 * max_cols + col], t);
    if (!b.is_cs && s[b.header_size + 16u * (uint32_t)col + 1u] == COL_RLE) {
      const uint32_t off = ld32(s, b.header_size + 16u * (uint32_t)col + 8u);
      if (off <= b.size && b.meta_off <= b.size - off && b.meta_off + off + 10u <= b.size)
        atomicMax(&col_span[4 * max_cols + col], (uint32_t)ld_bytes(s, b.meta_off + off + 2u, 4));
    }
  }
}

// Header survey of a device-resident image opened without a host view: one thread per block parses the
// 64-byte header (ObMicroBlockHeader::is_valid, ob_micro_block_header.cpp:53-61) and reports
// {row count, column count, verdict}: 0 ok, 1 invalid data, 2 not handled by the device path.
__global__ void __launch_bounds__(256) obgpu_survey_kernel(const uint8_t *image, const uint64_t *blk_off, const uint32_t *blk_size,
                                                           int n_blocks, uint32_t *out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_blocks) return;
  const uint8_t *s = image + blk_off[i];
  const uint32_t size = blk_size[i];
  const uint32_t w0 = ld32(s, 0);
  const int16_t magic = (int16_t)(w0 & 0xffff), version = (int16_t)(w0 >> 16);
  const uint32_t header_size = ld32(s, 4);
  const uint32_t ncol = ld32(s, 8) >> 16, nkey = ld32(s, 12) & 0xffffu;
  const uint32_t rows = ld32(s, 16);
  const uint32_t rst = ld32(s, 20) & 0xffu;
  const uint32_t row_data_off = ld32(s, 24);
  uint32_t verdict = 0;
  if (magic != MICRO_BLOCK_HEADER_MAGIC || version < 1 || version > 3 || ncol < nkey || rst >= MAX_ROW_STORE) verdict = 1;
  else if (rst != ENCODING_ROW_STORE && rst != SELECTIVE_ENCODING_ROW_STORE && rst != CS_ENCODING_ROW_STORE) verdict = 2;
  else {
    const bool is_cs = rst == CS_ENCODING_ROW_STORE;
    if (header_size < 64 || (uint64_t)header_size + (is_cs ? 12ull + 4ull * ncol : 16ull * ncol) > size ||
        (!is_cs && row_data_off > size) || rows == 0)
      verdict = 1;
    else if (rows > 65535u) verdict = 2;
  }
  out[2 * i] = rows;
  out[2 * i + 1] = ncol | (verdict << 16);
}

// =================================================================================================
// Count kernel: ONE WARP per micro-block evaluates the filter reading only the filter columns,
// straight from global memory (coalesced: 32 consecutive rows of a bit-packed column are one or two
// sectors), writes the packed selection bitmap and the block's selected-row count. No staging, no
// CTA barriers, no inter-block dependency.
// =================================================================================================
__global__ void __launch_bounds__(kThreads) obgpu_count_kernel(const __grid_constant__ ScanParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int block = blockIdx.x * kWarps + warp;
  if (block >= p.n_blocks) return;
  uint8_t *wr = g_smem + (uint32_t)warp * p.cw_bytes;
  ColDesc *descs = reinterpret_cast<ColDesc *>(wr + p.cw_desc);
  uint32_t *bm = reinterpret_cast<uint32_t *>(wr + p.cw_bm);
  uint32_t *bitsets = reinterpret_cast<uint32_t *>(wr + p.cw_bitset);
  Team t;
  t.tid = lane; t.nthreads = 32; t.warp = 0; t.nwarps = 1; t.lane = lane; t.bar_id = -1;

  const BlockRec rec = p.recs[block];
  const uint32_t rows = rec.rows;
  uint32_t *gbm = p.bitmap_words + rec.bm_word_off;
  if (p.blk_const != nullptr && rows != 0) {
    // the skip index decided this block (ObMicroIndexInfo::is_filter_always_false / _true): it is not read
    const uint8_t verdict = p.blk_const[block];
    if (verdict != 0) {
      const uint32_t nw = (rows + 31u) >> 5;
      for (uint32_t g = (uint32_t)lane; g < nw; g += 32u) gbm[g] = verdict == 1 ? valid_mask_of(rows, g) : 0u;
      if (lane == 0) p.counts[block] = verdict == 1 ? rows : 0u;
      return;
    }
  }
  bool bad = rows == 0;
  if (lane < p.n_used && p.used_in_filter[lane]) {
    const ColDesc d = p.plans[(int64_t)block * p.max_cols + p.used_col[lane]];
    descs[lane] = d;  // rle_slot stays -1: RLE filter columns use the run binary search here
    bad = bad || !d.ok;
  }
  const bool any_bad = __any_sync(0xffffffffu, bad);
  if (any_bad) {
    if (lane == 0) {
      atomicOr(p.status, rows == 0 ? ST_CORRUPT : ST_UNSUPPORTED);
      p.counts[block] = 0;
    }
    return;
  }
  BlockCtx c;
  const uint8_t *gblk = p.image + rec.off;
  view_from_rec(rec, gblk, c.b);
  c.sbit = 0;
  c.descs = descs;
  c.bitsets = bitsets;
  c.rle_base = nullptr;
  c.rle_slot_bytes = 0;
  c.rle_starts_bytes = 0;
  const uint32_t nwords = (rows + 31u) >> 5;
  __syncwarp();
  if (p.n_slots > 0 && p.simple_shape == 0) {
    for (int i = 0; i < p.n_nodes; ++i) {
      const FilterNodeDev &nd = p.nodes[i];
      if (nd.kind != NODE_WHITE || nd.slot < 0) continue;
      const ColDesc &d = descs[nd.used_idx];
      if (is_dict_kind(d))
        build_dict_bitset(p, c.b, d, nd, bitsets + nd.slot * p.bitset_words, t);
    }
    __syncwarp();
  }
  uint32_t cnt = 0;
  if (p.simple_shape != 0) {
    const bool and_mode = p.simple_shape == 1;
    const int n_leaves = p.n_nodes == 1 ? 1 : p.n_nodes - 1;
    uint8_t *stage = wr + p.cw_stage;
    bool inited = false;
    int staged_idx = -1;  // used-column index currently held by the staging buffer
    BlockCtx cs = c;
    for (int i = 0; i < n_leaves; ++i) {
      const FilterNodeDev &nd = p.nodes[i];
      const ColDesc &d = descs[nd.used_idx];
      // a leaf the skip index found constant on this (undecided) block is the neutral element of the AND / OR
      if (p.leaf_const != nullptr && p.leaf_const[(int64_t)block * p.n_nodes + i] != 0) continue;
      // stage the leaf column's region (ext bits, values / refs, run arrays, dictionary): every lane
      // pulls 16-byte pieces, 4 loads in flight per lane; all later reads hit shared memory
      bool staged = staged_idx == nd.used_idx;
      if (!staged && p.cw_stage_bytes > 0 && nd.op != OP_FALSE && nd.op != OP_TRUE) {
        uint32_t lo, hi;
        if (col_region(d, c.b, lo, hi) && hi - lo <= p.cw_stage_bytes && hi > lo) {
          const uint4 *src = reinterpret_cast<const uint4 *>(gblk + lo);
          uint4 *dst = reinterpret_cast<uint4 *>(stage);
          const uint32_t n16 = (hi - lo) >> 4;
          __syncwarp();
          for (uint32_t k = (uint32_t)lane; k < n16; k += 128u) {
            uint4 v0 = src[k], v1{}, v2{}, v3{};
            if (k + 32u < n16) v1 = src[k + 32u];
            if (k + 64u < n16) v2 = src[k + 64u];
            if (k + 96u < n16) v3 = src[k + 96u];
            dst[k] = v0;
            if (k + 32u < n16) dst[k + 32u] = v1;
            if (k + 64u < n16) dst[k + 64u] = v2;
            if (k + 96u < n16) dst[k + 96u] = v3;
          }
          __syncwarp();
          cs.b.s = stage - lo;  // block-relative offsets inside [lo, hi) now resolve to shared memory
          cs.sbit = (smem_u32(stage) - lo) * 8u;
          staged = true;
          staged_idx = nd.used_idx;
        } else {
          staged_idx = -1;
        }
      }
      if (nd.slot >= 0 && is_dict_kind(d)) {
        build_dict_bitset(p, staged ? cs.b : c.b, d, nd, bitsets + nd.slot * p.bitset_words, t);
        __syncwarp();
      }
      if (i == 0) {
        const bool fast = staged ? leaf_first_fast<false>(p, cs, nd, bm, rows, nwords, t)
                                 : leaf_first_fast<true>(p, c, nd, bm, rows, nwords, t);
        if (fast) {
          inited = true;
          __syncwarp();
          continue;
        }
      }
      if (!inited) {
        for (uint32_t g = (uint32_t)lane; g < nwords; g += 32u) bm[g] = and_mode ? valid_mask_of(rows, g) : 0u;
        inited = true;
        __syncwarp();
      }
      if (staged) leaf_over_words<false>(p, cs, nd, bm, rows, nwords, and_mode, t);
      else leaf_over_words<true>(p, c, nd, bm, rows, nwords, and_mode, t);
      __syncwarp();
      if (i + 1 < n_leaves) {
        // the reference's early-out (ob_pushdown_filter.cpp:1603-1615): AND stops once the bitmap is
        // all-false, OR once it is all-true
        bool undecided = false;
        for (uint32_t g = (uint32_t)lane; g < nwords; g += 32u)
          undecided = undecided || (and_mode ? bm[g] != 0u : bm[g] != valid_mask_of(rows, g));
        if (!__any_sync(0xffffffffu, undecided)) break;
      }
    }
    if (!inited) {  // every leaf was constant (cannot happen for an undecided block; kept for safety)
      for (uint32_t g = (uint32_t)lane; g < nwords; g += 32u) bm[g] = and_mode ? valid_mask_of(rows, g) : 0u;
      __syncwarp();
    }
    for (uint32_t g = (uint32_t)lane; g < nwords; g += 32u) {
      const uint32_t w = bm[g];
      gbm[g] = w;
      cnt += __popc(w);
    }
  } else {
    for (uint32_t g = 0; g < nwords; ++g) {
      const uint32_t row = g * 32u + (uint32_t)lane;
      const bool pr = row < rows && eval_tree(p, c, row);
      const uint32_t w = __ballot_sync(0xffffffffu, pr);
      if (lane == 0) {
        gbm[g] = w;
        cnt += __popc(w);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) p.counts[block] = cnt;
}

// =================================================================================================
// Prefix kernels: exclusive scan of the per-block counts -> sel_offset[n + 1].
//   pass 1: every CTA scans a 2048-element chunk (coalesced) and writes its total;
//   pass 2: every CTA adds the sum of the preceding chunk totals to its chunk.
// =================================================================================================
constexpr int kPrefixChunk = 2048;
__global__ void __launch_bounds__(256) obgpu_prefix_local_kernel(const uint32_t *counts, int n, int64_t *sel_offset,
                                                                 unsigned long long *chunk_total) {
  __shared__ unsigned long long s_warp[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int base = blockIdx.x * kPrefixChunk + tid * 8;
  uint32_t v[8];
  unsigned long long sum = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    v[k] = base + k < n ? counts[base + k] : 0u;
    sum += v[k];
  }
  unsigned long long inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long u = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += u;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  unsigned long long woff = 0, total = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    woff += k < warp ? s_warp[k] : 0ull;
    total += s_warp[k];
  }
  unsigned long long run = woff + inc - sum;
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    if (base + k < n) sel_offset[base + k] = (int64_t)run;
    run += v[k];
  }
  if (tid == 0) chunk_total[blockIdx.x] = total;
}

__global__ void __launch_bounds__(256) obgpu_prefix_fix_kernel(int n, int n_chunks, int64_t *sel_offset,
                                                               const unsigned long long *chunk_total) {
  __shared__ unsigned long long s_off;
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid < 32) {
    unsigned long long acc = 0;
    const int upto = blockIdx.x < n_chunks ? blockIdx.x : n_chunks;
    for (int k = lane; k < upto; k += 32) acc += chunk_total[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) s_off = acc;
  }
  __syncthreads();
  const unsigned long long off = s_off;
  if (blockIdx.x == n_chunks) {  // extra CTA: total
    if (tid == 0) sel_offset[n] = (int64_t)off;
    return;
  }
  const int base = blockIdx.x * kPrefixChunk + tid * 8;
#pragma unroll
  for (int k = 0; k < 8; ++k)
    if (base + k < n) sel_offset[base + k] += (int64_t)off;
}

// =================================================================================================
// Project kernel: one CTA (4 warps) per micro-block with at least one selected row. TMA stages the
// block while all warps turn the block's bitmap words into the ascending selected-row list. Then
// the projected COLUMNS are distributed over the warps (dynamic queue): a warp fetches the column's
// plan, builds its RLE run table if needed (warp-private scratch, no CTA barrier) and decodes every
// selected row of that column with coalesced stores at the dense offset given by the prefix.
// Per-column setup is thus paid by one warp instead of four, and a warp runs ~cnt/32 iterations per
// column instead of ~cnt/128.
// =================================================================================================
template <bool MULTI>
__global__ void __launch_bounds__(kThreads) obgpu_project_kernel(const __grid_constant__ ScanParams p) {
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ int s_next;
  __shared__ uint32_t s_scan[kWarps];
  __shared__ int32_t s_delta[kMaxProj];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint8_t *scr = g_smem + p.smem_scratch;
  uint16_t *sel = reinterpret_cast<uint16_t *>(scr + p.off_sel);
  uint32_t *bm = reinterpret_cast<uint32_t *>(scr + p.off_bm);
  uint32_t *wpre = reinterpret_cast<uint32_t *>(scr + p.off_wpre);
  // One block per CTA normally; with the sparse split most blocks belong to the warp-per-block kernel, so a CTA
  // walks p.proj_tiles consecutive blocks and only works on the dense ones (far fewer CTAs to launch and retire).
  // Blocks are visited last-to-first: the count kernel has just walked the batch front to back, so the
  // filter-column bytes of the LAST blocks are the ones still sitting in L2.
  bool used_bar = false;
  const int ntiles = MULTI ? p.proj_tiles : 1;  // MULTI = false: the loop and its bookkeeping compile away
  for (int it = 0; it < ntiles; ++it) {
    const int lin = (int)blockIdx.x * ntiles + it;
    if (lin >= p.n_blocks) break;
    const int tile = p.n_blocks - 1 - lin;
    if (used_bar) __syncthreads();  // everyone is done with the shared state of the previous block

    // one round trip: block record + the two prefix entries (independent loads)
    const BlockRec rec = p.recs[tile];
    const int64_t base = p.sel_offset[tile];
    const uint32_t cnt = (uint32_t)(p.sel_offset[tile + 1] - base);
    const uint32_t rows = rec.rows;
    if (rows == 0) {
      if (tid == 0) atomicOr(p.status, ST_CORRUPT);
      continue;
    }
    if (cnt == 0) continue;
    if (base + (int64_t)cnt > p.out_cap) {
      if (tid == 0) atomicOr(p.status, ST_OVERFLOW);
      continue;
    }
    // ---- second round trip, all in flight together: TMA of the block, the block's decode plans, the
    // first bitmap words ----------------------------------------------------------------------------------
    const uint32_t size = rec.size;
    // Few selected rows: staging the block would move far more bytes than the cells that are read. Such a
    // block is decoded straight from global memory (generic loads, a handful of sectors per column).
    const bool few = (uint64_t)cnt * 16u <= rows;
    if (few && p.sparse_split) continue;   // obgpu_project_sparse_kernel owns this block
    const bool sparse = few || p.no_stage != 0;
    if (tid == 0) {
      if (used_bar) mbar_inval(&s_bar);  // a block handled earlier by this CTA left the barrier initialised
      mbar_init(&s_bar, 1);
      fence_barrier_init();
      if (!p.compact && !sparse) {
        mbar_expect_tx(&s_bar, (size + 15u) & ~15u);
        tma_bulk_g2s(g_smem, p.image + rec.off, (size + 15u) & ~15u, &s_bar);
      }
      s_next = 0;
    }
    ColDesc *plans_s = reinterpret_cast<ColDesc *>(scr + p.off_plans);
    constexpr int kPieces = (int)(sizeof(ColDesc) / 16);
    const int npieces = p.n_proj * kPieces;
    uint4 pv0{}, pv1{};
    {
      const ColDesc *gp = p.plans + (int64_t)tile * p.max_cols;
      if (tid < npieces)
        pv0 = reinterpret_cast<const uint4 *>(gp + p.used_col[p.proj_used[tid / kPieces]])[tid % kPieces];
      if (tid + kThreads < npieces)
        pv1 = reinterpret_cast<const uint4 *>(gp + p.used_col[p.proj_used[(tid + kThreads) / kPieces]])[(tid + kThreads) % kPieces];
    }
    const uint32_t *gbm = p.bitmap_words + rec.bm_word_off;
    const bool all_rows = cnt == rows;
    const uint32_t nwords = (rows + 31u) >> 5;
    const uint32_t word0 = (!all_rows && (uint32_t)tid < nwords) ? gbm[tid] : 0u;
    if (tid < npieces) reinterpret_cast<uint4 *>(plans_s)[tid] = pv0;
    if (tid + kThreads < npieces) reinterpret_cast<uint4 *>(plans_s)[tid + kThreads] = pv1;
    __syncthreads();  // barrier object, queue and plans initialised before anyone uses them
    BlockCtx c;
    view_from_rec(rec, sparse ? p.image + rec.off : g_smem, c.b);
    if (p.compact && !sparse) {
      // Only the projected columns' regions are staged, packed back to back: lane pc of warp 0 issues
      // the bulk copy of column pc; s_delta[pc] = (offset in shared memory) - (offset in the block), so
      // block-relative addressing keeps working once the base is shifted by it.
      if (warp == 0) {
        uint32_t lo = 0, hi = 0;
        bool ok = false, var = false;
        if (lane < p.n_proj) {
          const ColDesc &d = plans_s[lane];
          ok = d.ok && col_region(d, c.b, lo, hi) && hi > lo;
          var = ok && d.kind == K_VARSTR;
        }
        // RAW var-length columns share one copy of the row data
        const uint32_t vmask = __ballot_sync(0xffffffffu, var);
        const int vfirst = __ffs(vmask) - 1;
        const bool dup = var && lane != vfirst;
        const uint32_t bytes = ok && !dup ? hi - lo : 0u;
        uint32_t inc = bytes;
  #pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += u;
        }
        uint32_t so = inc - bytes;
        const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
        const uint32_t vso = __shfl_sync(0xffffffffu, so, vfirst < 0 ? 0 : vfirst);
        if (dup) so = vso;
        if (lane < p.n_proj) s_delta[lane] = (int32_t)so - (int32_t)lo;
        if (lane == 0) mbar_expect_tx(&s_bar, total);
        __syncwarp();
        if (bytes) tma_bulk_g2s(g_smem + so, p.image + rec.off + lo, bytes, &s_bar);
      }
    }
    // ---- bitmap words -> popcount prefix -> ascending selected-row list (overlaps the TMA) ------------------
    if (!all_rows) {
      uint32_t run_total = 0;
      for (uint32_t base_w = 0; base_w < nwords; base_w += kThreads) {  // one pass for <= 4096 rows
        const uint32_t w = base_w + (uint32_t)tid;
        const uint32_t word = base_w == 0 ? word0 : (w < nwords ? gbm[w] : 0u);
        if (w < nwords) bm[w] = word;
        const uint32_t local = __popc(word);
        uint32_t inc = local;
  #pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += u;
        }
        if (lane == 31) s_scan[warp] = inc;
        __syncthreads();
        uint32_t warp_off = run_total, total = run_total;
  #pragma unroll
        for (int k = 0; k < kWarps; ++k) {
          const uint32_t v = s_scan[k];
          warp_off += k < warp ? v : 0u;
          total += v;
        }
        if (w < nwords) wpre[w] = warp_off + inc - local;
        run_total = total;
        __syncthreads();
      }
      for (uint32_t g = (uint32_t)warp; g < nwords; g += kWarps) {
        const uint32_t word = bm[g];
        if ((word >> lane) & 1u) sel[wpre[g] + __popc(word & ((1u << lane) - 1u))] = (uint16_t)(g * 32u + lane);
      }
      __syncthreads();
    }
    if (all_rows && sparse) {  // unstaged block with every row selected: the global path walks an identity list
      for (uint32_t j = (uint32_t)tid; j < cnt; j += kThreads) sel[j] = (uint16_t)j;
      __syncthreads();
    }
    // ---- block landed ---------------------------------------------------------------------------------------
    if (!sparse) mbar_wait(&s_bar, 0);
    c.sbit = smem_u32(g_smem) * 8u;
    c.bitsets = nullptr;
    // warp-private scratch: [run values][RLE run table]
    uint8_t *wscr = scr + p.off_desc + (uint32_t)warp * p.pw_bytes;
    c.descs = plans_s;
    c.rle_base = wscr + p.pw_rle;
    c.rle_slot_bytes = 0;  // one table per warp: slot 0
    c.rle_starts_bytes = p.words_cap * 4u;

    if (p.want_row_ids) {
      int32_t *rid = p.row_ids + base;
      if (all_rows) for (uint32_t j = (uint32_t)tid; j < cnt; j += kThreads) rid[j] = (int32_t)j;
      else for (uint32_t j = (uint32_t)tid; j < cnt; j += kThreads) rid[j] = (int32_t)sel[j];
    }
    const uint64_t blk_addr = block_string_addr(p, tile, rec.off);
    Team t;  // one warp per column
    t.tid = lane; t.nthreads = 32; t.warp = 0; t.nwarps = 1; t.lane = lane; t.bar_id = -1;
    for (;;) {
      int pc = 0;
      if (lane == 0) pc = atomicAdd(&s_next, 1);
      pc = __shfl_sync(0xffffffffu, pc, 0);
      if (pc >= p.n_proj) break;
      ColDesc *wdesc = plans_s + pc;  // this column's plan: only this warp touches it
      const ColDesc &d = *wdesc;
      if (sparse) {
        if (!d.ok) {
          if (lane == 0) atomicOr(p.status, ST_UNSUPPORTED);
        } else if (d.sc == 5) {
          project_str_col<false>(p, c, d, pc, sel, cnt, base, blk_addr, t);
        } else if (d.elem_len == 8) {
          project_int_col_global<uint64_t>(p, c, d, pc, sel, cnt, base, t);
        } else if (d.elem_len == 4) {
          project_int_col_global<uint32_t>(p, c, d, pc, sel, cnt, base, t);
        } else {
          project_int_col_global<uint8_t>(p, c, d, pc, sel, cnt, base, t);
        }
        __syncwarp();
        continue;
      }
      if (p.compact) {  // rebase onto this column's staged region
        const int32_t delta = s_delta[pc];
        c.b.s = g_smem + delta;
        c.sbit = (smem_u32(g_smem) + (uint32_t)delta) * 8u;
      }
      project_column_staged(p, c, wdesc, pc, sel, cnt, base, blk_addr, all_rows, rows, wscr, t);
      __syncwarp();
    }
    used_bar = true;
  }
}

// =================================================================================================
// Sparse projection: ONE WARP per micro-block whose selection is at most 1/16 of its rows (launched next to
// obgpu_project_kernel when the caller's selectivity hint says most blocks will be sparse). No staging, no
// CTA barriers: bitmap words -> selected-row list (warp scan), then every projected column is decoded for the
// few selected rows with generic loads from global memory. Four times as many blocks in flight per CTA slot.
// =================================================================================================
__global__ void __launch_bounds__(kThreads) obgpu_project_sparse_kernel(const __grid_constant__ ScanParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile = blockIdx.x * kWarps + warp;
  if (tile >= p.n_blocks) return;
  const BlockRec rec = p.recs[tile];
  const int64_t base = p.sel_offset[tile];
  const uint32_t cnt = (uint32_t)(p.sel_offset[tile + 1] - base);
  const uint32_t rows = rec.rows;
  if (rows == 0 || cnt == 0 || (uint64_t)cnt * 16u > rows) return;  // dense / empty / corrupt: the CTA kernel's job
  if (base + (int64_t)cnt > p.out_cap) {
    if (lane == 0) atomicOr(p.status, ST_OVERFLOW);
    return;
  }
  const uint32_t sel_cap = p.rows_cap / 16u + 32u;
  uint8_t *wr = g_smem + (uint32_t)warp * (((sel_cap * 2u + 15u) & ~15u) + (uint32_t)sizeof(ColDesc));
  uint16_t *sel = reinterpret_cast<uint16_t *>(wr);
  ColDesc *wdesc = reinterpret_cast<ColDesc *>(wr + ((sel_cap * 2u + 15u) & ~15u));
  // bitmap words -> ascending selected-row list
  const uint32_t *gbm = p.bitmap_words + rec.bm_word_off;
  const uint32_t nwords = (rows + 31u) >> 5;
  uint32_t running = 0;
  for (uint32_t base_w = 0; base_w < nwords; base_w += 32u) {
    const uint32_t w = base_w + (uint32_t)lane;
    uint32_t word = w < nwords ? gbm[w] : 0u;
    const uint32_t local = __popc(word);
    uint32_t inc = local;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t u = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += u;
    }
    uint32_t at = running + inc - local;
    while (word) {
      const uint32_t bit = (uint32_t)__ffs((int)word) - 1u;
      sel[at++] = (uint16_t)(w * 32u + bit);
      word &= word - 1u;
    }
    running += __shfl_sync(0xffffffffu, inc, 31);
  }
  __syncwarp();
  if (p.want_row_ids) {
    int32_t *rid = p.row_ids + base;
    for (uint32_t j = (uint32_t)lane; j < cnt; j += 32u) rid[j] = (int32_t)sel[j];
  }
  BlockCtx c;
  view_from_rec(rec, p.image + rec.off, c.b);
  c.sbit = 0;
  c.bitsets = nullptr;
  c.descs = wdesc;
  c.rle_base = nullptr;
  c.rle_slot_bytes = c.rle_starts_bytes = 0;
  const uint64_t blk_addr = block_string_addr(p, tile, rec.off);
  Team t;
  t.tid = lane; t.nthreads = 32; t.warp = 0; t.nwarps = 1; t.lane = lane; t.bar_id = -1;
  for (int pc = 0; pc < p.n_proj; ++pc) {
    __syncwarp();
    {
      const uint4 *src = reinterpret_cast<const uint4 *>(p.plans + (int64_t)tile * p.max_cols + p.used_col[p.proj_used[pc]]);
      if (lane < (int)(sizeof(ColDesc) / 16)) reinterpret_cast<uint4 *>(wdesc)[lane] = src[lane];
    }
    __syncwarp();
    const ColDesc &d = *wdesc;
    if (!d.ok) {
      if (lane == 0) atomicOr(p.status, ST_UNSUPPORTED);
    } else if (d.sc == 5) {
      project_str_col<false>(p, c, d, pc, sel, cnt, base, blk_addr, t);
    } else if (d.elem_len == 8) {
      project_int_col_global<uint64_t>(p, c, d, pc, sel, cnt, base, t);
    } else if (d.elem_len == 4) {
      project_int_col_global<uint32_t>(p, c, d, pc, sel, cnt, base, t);
    } else {
      project_int_col_global<uint8_t>(p, c, d, pc, sel, cnt, base, t);
    }
  }
}

// =================================================================================================
// Single-block kernels for the reference-granularity entry points (one CTA, kThreads threads)
// =================================================================================================
// ObBitmap byte image of a filter tree over rows [start, start + count) of one block.
__global__ void __launch_bounds__(kThreads) obgpu_filter_block_kernel(const __grid_constant__ ScanParams p,
                                                                      int tile, int64_t start, int64_t count,
                                                                      uint8_t *out_bytes) {
  __shared__ __align__(8) uint64_t s_bar;
  const Team t = cta_team();
  uint32_t *bitsets = reinterpret_cast<uint32_t *>(g_smem + p.smem_bitset);
  ColDesc *descs = reinterpret_cast<ColDesc *>(g_smem + p.smem_desc);
  if (t.tid == 0) {
    mbar_init(&s_bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const uint32_t size = p.blk_size[tile];
  load_block(g_smem, p.image + p.blk_off[tile], (size + 15u) & ~15u, &s_bar, 0);
  BlockCtx c;
  c.bitsets = bitsets;
  bool corrupt;
  bool ok = prepare_block(p, 0, size, descs, g_smem + p.smem_rle, t, c, corrupt);
  if (ok && (start < 0 || start + count > (int64_t)c.b.row_count)) {
    ok = false;
    corrupt = true;
  }
  if (!ok) {
    if (t.tid == 0) atomicOr(p.status, corrupt ? ST_CORRUPT : ST_UNSUPPORTED);
    return;
  }
  for (int i = 0; i < p.n_nodes; ++i) {
    const FilterNodeDev &nd = p.nodes[i];
    if (nd.kind != NODE_WHITE || nd.slot < 0) continue;
    const ColDesc &d = descs[nd.used_idx];
    if (is_dict_kind(d))
      build_dict_bitset(p, c.b, d, nd, bitsets + nd.slot * p.bitset_words, t);
  }
  __syncthreads();
  for (int64_t i = t.tid; i < count; i += kThreads)
    out_bytes[i] = eval_tree(p, c, (uint32_t)(start + i)) ? 1 : 0;
}

// decode_vector of one column for caller-supplied row ids (ObVectorDecodeCtx shape).
__global__ void __launch_bounds__(kThreads) obgpu_project_block_kernel(
    const __grid_constant__ ScanParams p, int tile, const int32_t *row_ids, int64_t row_cap, int64_t vec_offset,
    void *data, int32_t *lens, uint32_t *nulls, int32_t elem_len) {
  __shared__ __align__(8) uint64_t s_bar;
  const Team t = cta_team();
  ColDesc *descs = reinterpret_cast<ColDesc *>(g_smem + p.smem_desc);
  if (t.tid == 0) {
    mbar_init(&s_bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  const uint32_t size = p.blk_size[tile];
  load_block(g_smem, p.image + p.blk_off[tile], (size + 15u) & ~15u, &s_bar, 0);
  BlockCtx c;
  c.bitsets = nullptr;
  bool corrupt;
  if (!prepare_block(p, 0, size, descs, g_smem + p.smem_rle, t, c, corrupt)) {
    if (t.tid == 0) atomicOr(p.status, corrupt ? ST_CORRUPT : ST_UNSUPPORTED);
    return;
  }
  const ColDesc &d = descs[0];
  if ((d.sc == 5) != (lens != nullptr) || (d.sc != 5 && d.elem_len != elem_len)) {
    if (t.tid == 0) atomicOr(p.status, ST_UNSUPPORTED);
    return;
  }
  RleTable rt{};
  const RleTable *rtp = nullptr;
  if (d.kind == K_RLE && d.rle_slot >= 0) {
    rt = c.rle_table(d.rle_slot);
    rtp = &rt;
  }
  const uint64_t blk_addr = block_string_addr(p, tile, p.blk_off[tile]);
  for (int64_t i = t.tid; i < row_cap; i += kThreads) {
    const int32_t r = row_ids[i];
    if (r < 0 || (uint32_t)r >= c.b.row_count) {
      atomicOr(p.status, ST_CORRUPT);
      continue;
    }
    const int64_t o = vec_offset + i;
    bool is_null;
    if (d.sc == 5) {
      uint32_t cell, len;
      str_cell(c.b, d, rtp, (uint32_t)r, cell, len, is_null);
      if (!is_null) {
        reinterpret_cast<uint64_t *>(data)[o] = blk_addr + cell;
        lens[o] = (int32_t)len;
      }
    } else {
      const uint64_t v = int_cell(c.b, d, rtp, (uint32_t)r, is_null);
      if (!is_null) {
        if (elem_len == 8) reinterpret_cast<uint64_t *>(data)[o] = v;
        else if (elem_len == 4) reinterpret_cast<uint32_t *>(data)[o] = (uint32_t)v;
        else reinterpret_cast<uint8_t *>(data)[o] = (uint8_t)v;
      }
    }
    if (is_null) {
      atomicOr(&nulls[o >> 5], 1u << (o & 31));
      p.has_null[0] = 1;
    }
  }
}

// ObBitmap::get_row_ids: ascending ids of set bytes in [from, to), at most `limit`.
__global__ void __launch_bounds__(kThreads) obgpu_bitmap_row_ids_kernel(const uint8_t *bytes, int64_t from,
                                                                        int64_t to, int64_t limit,
                                                                        int64_t id_offset, int32_t *row_ids,
                                                                        int64_t *out_count) {
  __shared__ uint32_t s_scan[kWarps];
  __shared__ long long s_running;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_running = 0;
  __syncthreads();
  for (int64_t base = from; base < to; base += kThreads) {
    const long long running = s_running;
    if (running >= limit) break;
    const int64_t i = base + tid;
    const bool set = i < to && bytes[i] != 0;
    const uint32_t word = __ballot_sync(0xffffffffu, set);
    if (lane == 0) s_scan[warp] = __popc(word);
    __syncthreads();
    uint32_t off = 0, total = 0;
    for (int k = 0; k < kWarps; ++k) {
      if (k < warp) off += s_scan[k];
      total += s_scan[k];
    }
    if (set) {
      const long long pos = running + off + __popc(word & ((1u << lane) - 1u));
      if (pos < limit) row_ids[pos] = (int32_t)(i - id_offset);
    }
    __syncthreads();
    if (tid == 0) s_running = running + total;
    __syncthreads();
  }
  if (tid == 0) *out_count = s_running < limit ? s_running : limit;
}

#include "scan_small.cuh"
#include "stream_codecs.cuh"
#include "mat_codecs.cuh"

// =================================================================================================
// Host side
// =================================================================================================
#define CUDA_TRY(ctx, expr)                                                                       \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) {                                                                     \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                           \
      return e__ == cudaErrorMemoryAllocation ? OBGPU_ALLOCATE_MEMORY_FAILED : OBGPU_ERR_SYS;     \
    }                                                                                             \
  } while (0)

#include "skip_index.cuh"

struct obgpu_ctx {
  int device = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  std::string err;
  int64_t launches = 0;
  int max_smem_optin = 0;
  int sm_count = 0;
  int *h_pinned = nullptr;  // small pinned staging (status, totals)
  // optional kernel timing: ring of CUDA event pairs recorded around each scan kernel launch
  bool profiling = false;
  static constexpr int kProfRing = 256;
  cudaEvent_t ev0[kProfRing] = {nullptr}, ev1[kProfRing] = {nullptr};
  int64_t prof_count = 0;
};

struct obgpu_batch {
  obgpu_ctx *ctx = nullptr;
  const uint8_t *d_image = nullptr;
  bool own_image = false;
  int64_t image_size = 0;
  int32_t n_blocks = 0;
  std::vector<int64_t> offsets, sizes;
  std::vector<uint32_t> row_count;
  std::vector<int32_t> col_count;
  std::vector<int64_t> bm_word_off;  // n + 1
  int64_t total_rows = 0;
  uint32_t max_block_bytes = 0, max_rows = 0, max_cols = 0;
  std::vector<uint32_t> col_max_dict;  // per store index: max dict count + 2 over blocks
  std::vector<uint8_t> col_types;      // per store index: ObObjType (0xff: differs between blocks)
  std::vector<uint32_t> col_max_rle;   // per store index: max RLE run count over blocks (0: never RLE)
  // device tables (one allocation)
  void *d_tables = nullptr;
  uint64_t *d_blk_off = nullptr;
  uint32_t *d_blk_size = nullptr;
  int64_t *d_bm_word_off = nullptr;
  int64_t *d_row_start = nullptr;  // n + 1: first row of each block (dense row order of the batch)
  // decode plans + row counts built by the index kernel at open
  ColDesc *d_plans = nullptr;
  uint32_t *d_rows = nullptr;
  BlockRec *d_recs = nullptr;
  std::vector<uint32_t> col_span;      // per store index: max staged bytes of the value / ref array
  std::vector<uint32_t> col_pspan;     // per store index: max bytes a projection stages (proj_ranges)
  // skip index: serialized aggregate rows of the blocks (obgpu_batch_set_agg_rows), [d_agg_off[b], d_agg_off[b + 1])
  uint8_t *d_agg = nullptr;
  int64_t *d_agg_off = nullptr;
  // CS stream codecs: blocks restated as RAW at open (stream_codecs.cuh); nullptr when nothing had to be decoded
  obcs::XformRec *d_xf = nullptr;
  int64_t restated_blocks = 0, decoded_streams = 0;
  std::vector<uint8_t> col_mat;        // per store index: 1 when some block rebuilt the column's strings at open (mat_codecs.cuh)
  int64_t materialised_cols = 0;   // (block, column) pairs whose strings were rebuilt at open (mat_codecs.cuh)
};

struct ResultCol {
  void *data = nullptr;
  int32_t *lens = nullptr;
  uint32_t *nulls = nullptr;
  int32_t elem_len = 8;
  int32_t is_string = 0;
  int32_t obj_type = 0;
};

struct obgpu_result {
  obgpu_batch *batch = nullptr;
  obgpu_ctx *ctx = nullptr;
  void *arena = nullptr;
  size_t arena_bytes = 0;
  int32_t n_proj = 0;
  ResultCol cols[kMaxProj];
  int32_t *d_has_null = nullptr;
  int32_t *d_status = nullptr;
  int64_t *d_sel_offset = nullptr;
  uint32_t *d_bitmap = nullptr;
  int32_t *d_row_ids = nullptr;
  int64_t cap = 0;
  bool info_valid = false;
  bool no_filter = false;
  unsigned long long *d_skip_counters = nullptr;  // [always-false blocks, always-true blocks]
  int64_t skip_false = 0, skip_true = 0;
  obgpu_result_info info{};
  int32_t has_null[kMaxProj] = {0};
  int32_t status = 0;
  uint64_t string_base = 0;   // of the scan spec: where projected string pointers were expressed (obgpu_result_fetch_strings undoes it)
};

static thread_local std::string g_last_global_err;

extern "C" {

const char *obgpu_version(void) { return "obgpu_scan 0.1 (sm_100a, cuda " "12.9" ")"; }

int obgpu_ctx_create(int device, obgpu_ctx **out) {
  if (!out) return OBGPU_INVALID_ARGUMENT;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
    g_last_global_err = "no usable CUDA device (this library has no CPU fallback)";
    return OBGPU_ERR_SYS;
  }
  obgpu_ctx *c = new (std::nothrow) obgpu_ctx();
  if (!c) return OBGPU_ALLOCATE_MEMORY_FAILED;
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete c;
    return OBGPU_ERR_SYS;
  }
  c->stream = c->own_stream;
  cudaDeviceGetAttribute(&c->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaMallocHost(&c->h_pinned, 4096);
  // keep freed result arenas in the stream-ordered pool: steady-state scans do no cudaMalloc
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  // opt in to the full shared-memory carve-out (dynamic limit = opt-in max - static usage)
  auto opt_in = [&](const void *fn) {
    cudaFuncAttributes fa{};
    if (cudaFuncGetAttributes(&fa, fn) != cudaSuccess) return false;
    return cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                c->max_smem_optin - (int)fa.sharedSizeBytes) == cudaSuccess;
  };
  const bool ok = opt_in((const void *)obgpu_count_kernel) && opt_in((const void *)obgpu_project_kernel<false>) && opt_in((const void *)obgpu_project_kernel<true>) &&
                  opt_in((const void *)obgpu_filter_block_kernel) && opt_in((const void *)obgpu_project_block_kernel) &&
                  opt_in((const void *)obgpu_count_pipe_kernel) && opt_in((const void *)obgpu_project_pipe_kernel);
  cudaGetLastError();  // do not leave a stale (non-sticky) error for later launch checks
  if (!ok) {
    g_last_global_err = "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed: not an sm_100a device?";
    obgpu_ctx_destroy(c);
    return OBGPU_ERR_SYS;
  }
  c->max_smem_optin -= 1024;  // head-room for the kernels' static shared memory
  *out = c;
  return OBGPU_SUCCESS;
}

void obgpu_ctx_destroy(obgpu_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  if (ctx->h_pinned) cudaFreeHost(ctx->h_pinned);
  for (int i = 0; i < obgpu_ctx::kProfRing; ++i) {
    if (ctx->ev0[i]) cudaEventDestroy(ctx->ev0[i]);
    if (ctx->ev1[i]) cudaEventDestroy(ctx->ev1[i]);
  }
  delete ctx;
}

int obgpu_ctx_set_stream(obgpu_ctx *ctx, void *cuda_stream) {
  if (!ctx) return OBGPU_INVALID_ARGUMENT;
  ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
  return OBGPU_SUCCESS;
}

int obgpu_ctx_synchronize(obgpu_ctx *ctx) {
  if (!ctx) return OBGPU_INVALID_ARGUMENT;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

const char *obgpu_ctx_last_error(const obgpu_ctx *ctx) {
  return ctx ? ctx->err.c_str() : g_last_global_err.c_str();
}

int64_t obgpu_ctx_launch_count(const obgpu_ctx *ctx) { return ctx ? ctx->launches : 0; }

int obgpu_ctx_set_profiling(obgpu_ctx *ctx, int32_t enable) {
  if (!ctx) return OBGPU_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  if (enable && !ctx->ev0[0]) {
    for (int i = 0; i < obgpu_ctx::kProfRing; ++i) {
      CUDA_TRY(ctx, cudaEventCreate(&ctx->ev0[i]));
      CUDA_TRY(ctx, cudaEventCreate(&ctx->ev1[i]));
    }
  }
  ctx->profiling = enable != 0;
  ctx->prof_count = 0;
  return OBGPU_SUCCESS;
}

int obgpu_ctx_kernel_times(obgpu_ctx *ctx, float *ms, int32_t cap, int32_t *n) {
  if (!ctx || !ms || !n || cap < 0) return OBGPU_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const int64_t have = std::min<int64_t>(ctx->prof_count, obgpu_ctx::kProfRing);
  const int64_t take = std::min<int64_t>(have, cap);
  for (int64_t k = 0; k < take; ++k) {
    const int64_t idx = (ctx->prof_count - take + k) % obgpu_ctx::kProfRing;
    CUDA_TRY(ctx, cudaEventElapsedTime(&ms[k], ctx->ev0[idx], ctx->ev1[idx]));
  }
  *n = (int32_t)take;
  return OBGPU_SUCCESS;
}

// ---- batch ------------------------------------------------------------------------------------
// CS blocks with non-RAW integer streams -> a RAW restatement of the batch's image (stream_codecs.cuh), in place of
// the caller's image for every later kernel. Runs on the ctx stream after the image is resident; synchronises.
static int cs_restate_batch(obgpu_ctx *ctx, obgpu_batch *b) {
  const int32_t n = b->n_blocks;
  uint32_t *d_sv = nullptr;
  std::vector<uint32_t> sv((size_t)n * 4);
  CUDA_TRY(ctx, cudaMallocAsync((void **)&d_sv, (size_t)n * 16, ctx->stream));
  obcs::cs_survey_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, b->d_blk_off, b->d_blk_size, n, d_sv);
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(sv.data(), d_sv, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFreeAsync(d_sv, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return OBGPU_ERR_SYS; }
  bool any = false;
  for (int32_t i = 0; i < n; ++i) {
    const uint32_t flags = sv[(size_t)4 * i + 2];
    if (flags & obcs::XF_CORRUPT) { ctx->err = "corrupt CS micro block (stream layout)"; return OBGPU_INVALID_DATA; }
    if (flags & obcs::XF_UNSUPPORTED) continue;   // the index kernel marks the plans of such blocks unsupported: scans say OB_NOT_SUPPORTED
    any = any || (flags & obcs::XF_NONRAW);
  }
  if (!any) return OBGPU_SUCCESS;
  // layout of the restated image and of the job / scratch tables
  std::vector<uint64_t> tab((size_t)n * 3);   // [new_off][job_base][scratch_base]
  std::vector<uint32_t> nsz((size_t)n);
  uint64_t pos = 0, jobs = 0, scr = 0;
  int64_t restated = 0;
  for (int32_t i = 0; i < n; ++i) {
    const bool bad = (sv[(size_t)4 * i + 2] & obcs::XF_UNSUPPORTED) != 0;
    const uint32_t ns = bad ? (uint32_t)b->sizes[(size_t)i] : sv[(size_t)4 * i];
    tab[(size_t)i] = pos;
    tab[(size_t)n + i] = jobs;
    tab[(size_t)2 * n + i] = scr;
    nsz[(size_t)i] = ns;
    pos += ((uint64_t)ns + 127) & ~127ull;
    jobs += bad ? 0 : sv[(size_t)4 * i + 1];
    scr += 4ull * sv[(size_t)4 * i + 3];
    restated += (sv[(size_t)4 * i + 2] & obcs::XF_NONRAW) ? 1 : 0;
  }
  uint8_t *d_new = nullptr, *d_scr = nullptr;
  uint64_t *d_tab = nullptr;
  uint32_t *d_nsz = nullptr;
  obcs::StreamJob *d_jobs = nullptr;
  int *d_status = nullptr;
  auto cleanup = [&]() {
    if (d_scr) cudaFreeAsync(d_scr, ctx->stream);
    if (d_tab) cudaFreeAsync(d_tab, ctx->stream);
    if (d_nsz) cudaFreeAsync(d_nsz, ctx->stream);
    if (d_jobs) cudaFreeAsync(d_jobs, ctx->stream);
    if (d_status) cudaFreeAsync(d_status, ctx->stream);
  };
  e = cudaMallocAsync((void **)&d_new, (size_t)pos + 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_scr, (size_t)scr + 16, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_tab, (size_t)n * 24, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_nsz, (size_t)n * 4, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_jobs, (size_t)(jobs + 1) * sizeof(obcs::StreamJob), ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_status, 16, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&b->d_xf, (size_t)n * sizeof(obcs::XformRec), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_status, 0, 16, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_new, 0, (size_t)pos + 64, ctx->stream);   // block padding and tail slack read as zero
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab, tab.data(), (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_nsz, nsz.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    obcs::cs_rewrite_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, b->d_blk_off, b->d_blk_size, n, d_new, d_tab, d_nsz,
                                                                              d_tab + n, d_jobs, d_scr, d_tab + 2 * (size_t)n, b->d_xf, d_status);
    if (jobs > 0)
      obcs::cs_decode_kernel<<<(unsigned)((jobs + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, d_new, d_jobs, (int64_t)jobs, d_status);
    ctx->launches += jobs > 0 ? 2 : 1;
    e = cudaGetLastError();
  }
  int st = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(&st, d_status, 4, cudaMemcpyDeviceToHost, ctx->stream);
  // the batch now lives in the restated image
  if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_blk_off, tab.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_blk_size, nsz.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cleanup();
  if (e != cudaSuccess || st != 0) {
    if (d_new) cudaFreeAsync(d_new, ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return e == cudaErrorMemoryAllocation ? OBGPU_ALLOCATE_MEMORY_FAILED : OBGPU_ERR_SYS; }
    ctx->err = "CS integer stream does not decode (corrupt or unsupported codec)";
    return (st & obcs::XF_CORRUPT) ? OBGPU_INVALID_DATA : OBGPU_NOT_SUPPORTED;
  }
  if (b->own_image && b->d_image) cudaFreeAsync((void *)b->d_image, ctx->stream);
  b->d_image = d_new;
  b->own_image = true;
  b->image_size = (int64_t)pos;
  b->max_block_bytes = 0;
  for (int32_t i = 0; i < n; ++i) {
    b->offsets[(size_t)i] = (int64_t)tab[(size_t)i];
    b->sizes[(size_t)i] = nsz[(size_t)i];
    b->max_block_bytes = std::max<uint32_t>(b->max_block_bytes, (nsz[(size_t)i] + 15u) & ~15u);
  }
  b->restated_blocks = restated;
  b->decoded_streams = (int64_t)jobs;
  return OBGPU_SUCCESS;
}

// PAX blocks with HEX_PACKING / STRING_DIFF / STRING_PREFIX columns -> a copy of the batch's image in which every such column has
// its strings materialised behind the block (mat_codecs.cuh). Runs after cs_restate_batch (the two compose: a batch may hold both
// kinds of blocks); synchronises.
static int pax_materialise_batch(obgpu_ctx *ctx, obgpu_batch *b) {
  const int32_t n = b->n_blocks;
  uint32_t *d_flag = nullptr;
  uint32_t flag = 0;
  CUDA_TRY(ctx, cudaMallocAsync((void **)&d_flag, 16, ctx->stream));
  cudaError_t e = cudaMemsetAsync(d_flag, 0, 16, ctx->stream);
  if (e == cudaSuccess) {
    obmat::mat_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(b->d_image, b->d_blk_off, b->d_blk_size, n, d_flag);
    ctx->launches++;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFreeAsync(d_flag, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return OBGPU_ERR_SYS; }
  if (!(flag & obmat::MF_ANY)) return OBGPU_SUCCESS;
  uint32_t *d_sv = nullptr;
  std::vector<uint32_t> sv((size_t)n * 4);
  CUDA_TRY(ctx, cudaMallocAsync((void **)&d_sv, (size_t)n * 16, ctx->stream));
  obmat::mat_survey_kernel<<<(unsigned)(((int64_t)n * 32 + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, b->d_blk_off, b->d_blk_size, n, d_sv);
  ctx->launches++;
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(sv.data(), d_sv, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFreeAsync(d_sv, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return OBGPU_ERR_SYS; }
  std::vector<uint64_t> tab((size_t)n * 2);   // [new_off][job_base]
  std::vector<uint32_t> nsz((size_t)n);
  uint64_t pos = 0, jobs = 0;
  for (int32_t i = 0; i < n; ++i) {
    tab[(size_t)i] = pos;
    tab[(size_t)n + i] = jobs;
    nsz[(size_t)i] = sv[(size_t)4 * i];
    pos += ((uint64_t)sv[(size_t)4 * i] + 127) & ~127ull;
    jobs += sv[(size_t)4 * i + 1];
  }
  if (jobs == 0) return OBGPU_SUCCESS;   // every such column was refused: the index kernel leaves them unsupported
  uint8_t *d_new = nullptr;
  uint64_t *d_tab = nullptr;
  uint32_t *d_nsz = nullptr;
  obmat::MatJob *d_jobs = nullptr;
  int *d_status = nullptr;
  obcs::XformRec *d_xf = nullptr;
  std::vector<obcs::XformRec> xf((size_t)n);
  auto cleanup = [&]() {
    if (d_tab) cudaFreeAsync(d_tab, ctx->stream);
    if (d_nsz) cudaFreeAsync(d_nsz, ctx->stream);
    if (d_jobs) cudaFreeAsync(d_jobs, ctx->stream);
    if (d_status) cudaFreeAsync(d_status, ctx->stream);
  };
  // where the caller's image has every block (string pointers of the untouched columns keep addressing it): carried over from
  // the CS restatement when that ran
  if (b->d_xf) {
    e = cudaMemcpyAsync(xf.data(), b->d_xf, (size_t)n * sizeof(obcs::XformRec), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return OBGPU_ERR_SYS; }
  } else {
    for (int32_t i = 0; i < n; ++i) { xf[(size_t)i].orig_off = (uint64_t)b->offsets[(size_t)i]; xf[(size_t)i].str_delta = 0; }
  }
  e = cudaMallocAsync((void **)&d_new, (size_t)pos + 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_tab, (size_t)n * 16, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_nsz, (size_t)n * 4, ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_jobs, (size_t)(jobs + 1) * sizeof(obmat::MatJob), ctx->stream);
  if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_status, 16, ctx->stream);
  if (e == cudaSuccess && !b->d_xf) e = cudaMallocAsync((void **)&d_xf, (size_t)n * sizeof(obcs::XformRec), ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_status, 0, 16, ctx->stream);
  if (e == cudaSuccess) e = cudaMemsetAsync(d_new, 0, (size_t)pos + 64, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab, tab.data(), (size_t)n * 16, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_nsz, nsz.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    obmat::mat_rewrite_kernel<<<(unsigned)(((int64_t)n * 32 + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, b->d_blk_off, b->d_blk_size, n, d_new,
                                                                                             d_tab, d_nsz, d_tab + n, d_jobs);
    obmat::mat_decode_kernel<<<(unsigned)(((int64_t)jobs * 32 + 127) / 128), 128, 0, ctx->stream>>>(b->d_image, d_new, d_jobs, (int64_t)jobs, d_status);
    ctx->launches += 2;
    e = cudaGetLastError();
  }
  int st = 0;
  if (e == cudaSuccess) e = cudaMemcpyAsync(&st, d_status, 4, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_blk_off, tab.data(), (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_blk_size, nsz.data(), (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess && d_xf) e = cudaMemcpyAsync(d_xf, xf.data(), (size_t)n * sizeof(obcs::XformRec), cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cleanup();
  if (e != cudaSuccess || st != 0) {
    if (d_new) cudaFreeAsync(d_new, ctx->stream);
    if (d_xf) cudaFreeAsync(d_xf, ctx->stream);
    if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return e == cudaErrorMemoryAllocation ? OBGPU_ALLOCATE_MEMORY_FAILED : OBGPU_ERR_SYS; }
    ctx->err = "HEX_PACKING / STRING_DIFF / STRING_PREFIX column does not decode (corrupt micro block)";
    return OBGPU_INVALID_DATA;
  }
  if (b->own_image && b->d_image) cudaFreeAsync((void *)b->d_image, ctx->stream);
  b->d_image = d_new;
  b->own_image = true;
  b->image_size = (int64_t)pos;
  if (d_xf) b->d_xf = d_xf;
  b->max_block_bytes = 0;
  for (int32_t i = 0; i < n; ++i) {
    b->offsets[(size_t)i] = (int64_t)tab[(size_t)i];
    b->sizes[(size_t)i] = nsz[(size_t)i];
    b->max_block_bytes = std::max<uint32_t>(b->max_block_bytes, (nsz[(size_t)i] + 15u) & ~15u);
  }
  b->materialised_cols = (int64_t)jobs;
  return OBGPU_SUCCESS;
}

static uint32_t rd32h(const uint8_t *p) { uint32_t v; memcpy(&v, p, 4); return v; }
static uint16_t rd16h(const uint8_t *p) { uint16_t v; memcpy(&v, p, 2); return v; }

int obgpu_batch_open(obgpu_ctx *ctx, const void *image, int64_t image_size, const int64_t *offsets,
                     const int64_t *sizes, int32_t n_blocks, int32_t image_on_device, const void *header_view,
                     obgpu_batch **out) {
  if (!ctx || !image || !offsets || !sizes || n_blocks <= 0 || !out || image_size <= 0)
    return OBGPU_INVALID_ARGUMENT;
  // header facts come from a host view of the blocks when there is one; a device-resident image opened without
  // a host view is surveyed on the device instead (obgpu_survey_kernel)
  const uint8_t *host = image_on_device ? (const uint8_t *)header_view : (const uint8_t *)image;
  if (image_on_device && ((uintptr_t)image & 15u) != 0) {
    ctx->err = "device-resident image must be 16-byte aligned (TMA bulk copies)";
    return OBGPU_INVALID_ARGUMENT;
  }
  cudaSetDevice(ctx->device);
  obgpu_batch *b = new (std::nothrow) obgpu_batch();
  if (!b) return OBGPU_ALLOCATE_MEMORY_FAILED;
  b->ctx = ctx;
  b->n_blocks = n_blocks;
  b->image_size = image_size;
  b->offsets.assign(offsets, offsets + n_blocks);
  b->sizes.assign(sizes, sizes + n_blocks);
  b->row_count.resize((size_t)n_blocks);
  b->col_count.resize((size_t)n_blocks);
  b->bm_word_off.resize((size_t)n_blocks + 1);
  int ret = OBGPU_SUCCESS;
  bool any_cs = false, any_mat = false;
  for (int32_t i = 0; i < n_blocks; ++i) {
    const int64_t off = offsets[i], sz = sizes[i];
    if (off < 0 || (off & 15) || sz < 64 || sz > 0x7fffffffll || off + sz > image_size) { ret = OBGPU_INVALID_ARGUMENT; break; }
    const int64_t padded = (sz + 15) & ~15ll;
    const int64_t limit = i + 1 < n_blocks ? offsets[i + 1] : image_size;
    if (image_on_device && off + padded > limit) {
      ctx->err = "blocks of a device-resident image must be padded to 16 bytes";
      ret = OBGPU_INVALID_ARGUMENT;
      break;
    }
    b->max_block_bytes = std::max<uint32_t>(b->max_block_bytes, (uint32_t)padded);
  }
  if (ret != OBGPU_SUCCESS) { delete b; return ret; }
  // device tables: [blk_off u64 x n][bm_word_off i64 x (n + 1)][blk_size u32 x n] ... [row_start i64 x (n + 1)]
  const size_t tb_rs = (((size_t)n_blocks * (8 + 4) + ((size_t)n_blocks + 1) * 8) + 15) & ~(size_t)15;  // row_start follows
  const size_t tb = tb_rs + ((size_t)n_blocks + 1) * 8 + 64;
  cudaError_t e = cudaMallocAsync(&b->d_tables, tb, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); delete b; return OBGPU_ALLOCATE_MEMORY_FAILED; }
  uint8_t *dt = (uint8_t *)b->d_tables;
  b->d_blk_off = (uint64_t *)dt;
  b->d_bm_word_off = (int64_t *)(dt + (size_t)n_blocks * 8);
  b->d_blk_size = (uint32_t *)(dt + (size_t)n_blocks * 8 + ((size_t)n_blocks + 1) * 8);
  b->d_row_start = (int64_t *)(dt + tb_rs);
  std::vector<uint8_t> stage(tb);
  {
    uint64_t *o = (uint64_t *)stage.data();
    uint32_t *s = (uint32_t *)(stage.data() + (size_t)n_blocks * 8 + ((size_t)n_blocks + 1) * 8);
    for (int32_t i = 0; i < n_blocks; ++i) { o[i] = (uint64_t)offsets[i]; s[i] = (uint32_t)sizes[i]; }
  }
  if (host) {
    for (int32_t i = 0; i < n_blocks && ret == OBGPU_SUCCESS; ++i) {
      const int64_t sz = sizes[i];
      const uint8_t *p = host + offsets[i];
      const int16_t magic = (int16_t)rd16h(p), version = (int16_t)rd16h(p + 2);
      const uint32_t header_size = rd32h(p + 4);
      const uint16_t ncol = rd16h(p + 10), nkey = rd16h(p + 12);
      const uint32_t rows = rd32h(p + 16);
      const uint8_t rst = p[20];
      const uint32_t row_data_off = rd32h(p + 24);
      // ObMicroBlockHeader::is_valid (ob_micro_block_header.cpp:53-61) + get_micro_metas bounds
      if (magic != obf::MICRO_BLOCK_HEADER_MAGIC || version < 1 || version > 3 || ncol < nkey || rst >= obf::MAX_ROW_STORE) {
        ctx->err = "invalid micro block header";
        ret = OBGPU_INVALID_DATA;
        break;
      }
      const bool is_cs = rst == obf::CS_ENCODING_ROW_STORE;
      if (rst != obf::ENCODING_ROW_STORE && rst != obf::SELECTIVE_ENCODING_ROW_STORE && !is_cs) {
        ctx->err = "row store type not handled by the device path";
        ret = OBGPU_NOT_SUPPORTED;
        break;
      }
      if (header_size < 64 || (int64_t)header_size + (is_cs ? 12ll + 4ll * ncol : 16ll * ncol) > sz || (!is_cs && row_data_off > sz) ||
          rows == 0) {
        ret = OBGPU_INVALID_DATA;
        break;
      }
      if (rows > 65535u) {
        ctx->err = "more than 65535 rows in one micro block";
        ret = OBGPU_NOT_SUPPORTED;
        break;
      }
      b->row_count[(size_t)i] = rows;
      b->col_count[(size_t)i] = ncol;
      any_cs = any_cs || is_cs;
      if (!is_cs && !any_mat)
        for (uint32_t c = 0; c < ncol; ++c) {
          const uint8_t t = p[header_size + 16u * c + 1];
          if (t == obf::COL_STRING_DIFF || t == obf::COL_HEX_PACKING || t == obf::COL_STRING_PREFIX || t == obf::COL_COLUMN_EQUAL ||
              t == obf::COL_COLUMN_SUBSTR) {
            any_mat = true;
            break;
          }
        }
    }
  } else {
    any_cs = true;   // no host view: the survey kernel of the restatement looks at every block's store type
    any_mat = true;  // ... and the probe kernel of the materialisation at every block's column types
    if (!image_on_device) { ret = OBGPU_INVALID_ARGUMENT; }
    uint32_t *d_sv = nullptr;
    std::vector<uint32_t> sv((size_t)n_blocks * 2);
    if (ret == OBGPU_SUCCESS) {
      e = cudaMemcpyAsync(b->d_tables, stage.data(), tb_rs, cudaMemcpyHostToDevice, ctx->stream);
      if (e == cudaSuccess) e = cudaMallocAsync((void **)&d_sv, (size_t)n_blocks * 8, ctx->stream);
      if (e == cudaSuccess) {
        obgpu_survey_kernel<<<(unsigned)((n_blocks + 255) / 256), 256, 0, ctx->stream>>>((const uint8_t *)image, b->d_blk_off, b->d_blk_size,
                                                                                         n_blocks, d_sv);
        ctx->launches++;
        e = cudaGetLastError();
      }
      if (e == cudaSuccess) e = cudaMemcpyAsync(sv.data(), d_sv, (size_t)n_blocks * 8, cudaMemcpyDeviceToHost, ctx->stream);
      if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
      if (d_sv) cudaFreeAsync(d_sv, ctx->stream);
      if (e != cudaSuccess) {
        ctx->err = cudaGetErrorString(e);
        obgpu_batch_close(b);
        return e == cudaErrorMemoryAllocation ? OBGPU_ALLOCATE_MEMORY_FAILED : OBGPU_ERR_SYS;
      }
      for (int32_t i = 0; i < n_blocks; ++i) {
        const uint32_t verdict = sv[(size_t)2 * i + 1] >> 16;
        if (verdict != 0) {
          ctx->err = verdict == 1 ? "invalid micro block header" : "micro block not handled by the device path";
          ret = verdict == 1 ? OBGPU_INVALID_DATA : OBGPU_NOT_SUPPORTED;
          break;
        }
        b->row_count[(size_t)i] = sv[(size_t)2 * i];
        b->col_count[(size_t)i] = (int32_t)(sv[(size_t)2 * i + 1] & 0xffffu);
      }
    }
  }
  if (ret != OBGPU_SUCCESS) {
    obgpu_batch_close(b);
    return ret;
  }
  int64_t words = 0;
  for (int32_t i = 0; i < n_blocks; ++i) {
    const uint32_t rows = b->row_count[(size_t)i];
    b->bm_word_off[(size_t)i] = words;
    words += (rows + 31) / 32;
    b->total_rows += rows;
    b->max_rows = std::max(b->max_rows, rows);
    b->max_cols = std::max<uint32_t>(b->max_cols, (uint32_t)b->col_count[(size_t)i]);
  }
  b->bm_word_off[(size_t)n_blocks] = words;
  b->col_max_dict.assign(b->max_cols, 0);
  b->col_types.assign(b->max_cols, 0);
  b->col_max_rle.assign(b->max_cols, 0);
  // blocks larger than a shared-memory page are fine for the batch scan (columns are then decoded straight
  // from global memory); only the one-block entry points need the block to fit
  {
    int64_t *w = (int64_t *)(stage.data() + (size_t)n_blocks * 8);
    memcpy(w, b->bm_word_off.data(), ((size_t)n_blocks + 1) * 8);
    int64_t *rs = (int64_t *)(stage.data() + tb_rs);  // first row of every block in the batch's row order
    rs[0] = 0;
    for (int32_t i = 0; i < n_blocks; ++i) rs[i + 1] = rs[i] + b->row_count[(size_t)i];
  }
  e = cudaMemcpyAsync(b->d_tables, stage.data(), tb, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess) {
    if (image_on_device) {
      b->d_image = (const uint8_t *)image;
    } else {
      void *di = nullptr;
      e = cudaMallocAsync(&di, (size_t)image_size + 64, ctx->stream);
      if (e == cudaSuccess) {
        b->d_image = (const uint8_t *)di;
        b->own_image = true;
        e = cudaMemsetAsync((uint8_t *)di + image_size, 0, 64, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(di, image, (size_t)image_size, cudaMemcpyHostToDevice, ctx->stream);
      }
    }
  }
  // CS blocks whose integer streams carry codecs are restated as RAW once, here (the reference's full_transform at cache fill)
  if (e == cudaSuccess && any_cs) {
    const int rret = cs_restate_batch(ctx, b);
    if (rret != OBGPU_SUCCESS) {
      obgpu_batch_close(b);
      return rret;
    }
  }
  // PAX string codecs that rebuild their values (HEX_PACKING / STRING_DIFF / STRING_PREFIX): materialised once, here
  if (e == cudaSuccess && any_mat) {
    const int mret = pax_materialise_batch(ctx, b);
    if (mret != OBGPU_SUCCESS) {
      obgpu_batch_close(b);
      return mret;
    }
  }
  // decode plans: one thread per (block, column)
  if (e == cudaSuccess && b->max_cols > 128) {
    ctx->err = "more than 128 columns in a micro block";
    obgpu_batch_close(b);
    return OBGPU_NOT_SUPPORTED;
  }
  if (e == cudaSuccess) {
    const size_t plan_bytes = (size_t)n_blocks * b->max_cols * sizeof(ColDesc);
    void *dp = nullptr;
    const size_t rows_bytes = ((size_t)n_blocks * 4 + 63) & ~(size_t)63;
    const size_t rec_bytes = (size_t)n_blocks * sizeof(BlockRec);
    e = cudaMallocAsync(&dp, plan_bytes + rows_bytes + rec_bytes + (size_t)b->max_cols * 28 + 64, ctx->stream);
    if (e == cudaSuccess) {
      b->d_plans = (ColDesc *)dp;
      b->d_rows = (uint32_t *)((uint8_t *)dp + plan_bytes);
      b->d_recs = (BlockRec *)((uint8_t *)dp + plan_bytes + rows_bytes);
      uint32_t *d_span = (uint32_t *)((uint8_t *)dp + plan_bytes + rows_bytes + rec_bytes);
      // per-column reductions of the index kernel: [region span][dictionary size][type min][type max][RLE runs][projection span][materialised]
      e = cudaMemsetAsync(d_span, 0, (size_t)b->max_cols * 28, ctx->stream);
      if (e == cudaSuccess) e = cudaMemsetAsync(d_span + 2 * (size_t)b->max_cols, 0xff, (size_t)b->max_cols * 4, ctx->stream);
      const int64_t nthreads = (int64_t)n_blocks * b->max_cols;
      obgpu_index_kernel<<<(unsigned)((nthreads + 255) / 256), 256, 0, ctx->stream>>>(
          b->d_image, b->d_blk_off, b->d_blk_size, b->d_bm_word_off, n_blocks, (int)b->max_cols, b->d_plans,
          b->d_rows, b->d_recs, d_span);
      if (e == cudaSuccess) e = cudaGetLastError();
      ctx->launches++;
      b->col_span.assign((size_t)b->max_cols * 7, 0);
      if (e == cudaSuccess)
        e = cudaMemcpyAsync(b->col_span.data(), d_span, (size_t)b->max_cols * 28, cudaMemcpyDeviceToHost, ctx->stream);
    }
  }
  // `stage` is pageable: the copy above is staged synchronously by the runtime before returning
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  if (e == cudaSuccess && b->col_span.size() == (size_t)b->max_cols * 7) {
    const size_t mc = b->max_cols;
    b->col_pspan.assign(b->col_span.begin() + 5 * mc, b->col_span.begin() + 6 * mc);
    b->col_mat.assign(mc, 0);
    for (size_t c = 0; c < mc; ++c) b->col_mat[c] = b->col_span[6 * mc + c] ? 1 : 0;
    for (size_t c = 0; c < mc; ++c) {
      b->col_max_dict[c] = b->col_span[mc + c];
      const uint32_t tmin = b->col_span[2 * mc + c], tmax = b->col_span[3 * mc + c];
      b->col_types[c] = tmin == 0xffffffffu ? 0 : (tmin == tmax ? (uint8_t)tmin : 0xff);   // 0xff: the blocks disagree
      b->col_max_rle[c] = b->col_span[4 * mc + c];
    }
    b->col_span.resize(mc);
  }
  if (e != cudaSuccess) {
    ctx->err = cudaGetErrorString(e);
    obgpu_batch_close(b);
    return e == cudaErrorMemoryAllocation ? OBGPU_ALLOCATE_MEMORY_FAILED : OBGPU_ERR_SYS;
  }
  *out = b;
  return OBGPU_SUCCESS;
}

void obgpu_batch_close(obgpu_batch *b) {
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  if (b->d_tables) cudaFreeAsync(b->d_tables, b->ctx->stream);
  if (b->d_plans) cudaFreeAsync(b->d_plans, b->ctx->stream);
  if (b->d_agg) cudaFreeAsync(b->d_agg, b->ctx->stream);
  if (b->d_agg_off) cudaFreeAsync(b->d_agg_off, b->ctx->stream);
  if (b->d_xf) cudaFreeAsync(b->d_xf, b->ctx->stream);
  if (b->own_image && b->d_image) cudaFreeAsync((void *)b->d_image, b->ctx->stream);
  delete b;
}

int obgpu_batch_block_info(const obgpu_batch *b, int32_t block, int64_t *row_count, int32_t *column_count) {
  if (!b || block < 0 || block >= b->n_blocks) return OBGPU_INVALID_ARGUMENT;
  if (row_count) *row_count = b->row_count[(size_t)block];
  if (column_count) *column_count = b->col_count[(size_t)block];
  return OBGPU_SUCCESS;
}

int obgpu_batch_total_rows(const obgpu_batch *b, int64_t *total_rows) {
  if (!b || !total_rows) return OBGPU_INVALID_ARGUMENT;
  *total_rows = b->total_rows;
  return OBGPU_SUCCESS;
}

}  // extern "C"

// ---- building the kernel parameter block ---------------------------------------------------------
static int used_index(ScanParams &p, int32_t col) {
  for (int i = 0; i < p.n_used; ++i)
    if (p.used_col[i] == col) return i;
  if (p.n_used >= kMaxUsedCols) return -1;
  p.used_col[p.n_used] = col;
  return p.n_used++;
}

// Flattens / validates the filter; resolves NULL constants the way
// ObMicroBlockDecoder::filter_pushdown_filter does (ob_micro_block_decoder.cpp:1713-1715).
static int build_filter(obgpu_ctx *ctx, const obgpu_batch *b, const obgpu_filter *f, ScanParams &p) {
  p.n_nodes = 0;
  p.n_slots = 0;
  p.bitset_words = 0;
  p.simple_shape = 0;
  if (!f || f->n_nodes == 0) return OBGPU_SUCCESS;
  if (!f->nodes || f->n_nodes < 0 || f->n_nodes > kMaxNodes) {
    ctx->err = "filter tree too large for the device path";
    return f && f->n_nodes > kMaxNodes ? OBGPU_NOT_SUPPORTED : OBGPU_INVALID_ARGUMENT;
  }
  int n_params = 0;
  uint32_t heap = 0;
  int depth = 0;
  for (int i = 0; i < f->n_nodes; ++i) {
    const obgpu_filter_node &src = f->nodes[i];
    FilterNodeDev nd{};
    nd.kind = (int8_t)src.kind;
    nd.slot = -1;
    if (src.kind == OBGPU_NODE_WHITE) {
      if (src.op < 0 || src.op >= OBGPU_WHITE_OP_MAX || src.col < 0) return OBGPU_INVALID_ARGUMENT;
      const int np = src.n_params;
      if ((src.op <= OBGPU_WHITE_OP_NE && np != 1) || (src.op == OBGPU_WHITE_OP_BT && np != 2) ||
          (src.op == OBGPU_WHITE_OP_IN && np < 1) || (src.op >= OBGPU_WHITE_OP_NU && np != 0))
        return OBGPU_INVALID_ARGUMENT;
      if (np > 0 && (!f->params || src.param_begin < 0 || src.param_begin + np > f->n_params))
        return OBGPU_INVALID_ARGUMENT;
      const int ui = used_index(p, src.col);
      if (ui < 0) return OBGPU_NOT_SUPPORTED;
      if ((uint32_t)src.col >= b->max_cols) return OBGPU_INVALID_ARGUMENT;
      p.used_in_filter[ui] = 1;
      nd.used_idx = (int16_t)ui;
      nd.op = (int16_t)src.op;
      nd.param_begin = (int16_t)n_params;
      int kept = 0;
      bool null_param = false;
      for (int k = 0; k < np; ++k) {
        const obgpu_filter_param &sp = f->params[src.param_begin + k];
        if (sp.is_null) {
          if (src.op == OBGPU_WHITE_OP_IN) continue;  // NULLs never match inside an IN list
          null_param = true;
          continue;
        }
        if (n_params >= kMaxParams) return OBGPU_NOT_SUPPORTED;
        ParamDev pd{};
        pd.i64 = sp.i64;
        pd.len = sp.len;
        pd.heap_off = heap;
        if (sp.ptr && sp.len > 0) {
          // constants start 8-byte aligned and are padded to 8 bytes: str_cmp reads them in 64-bit words
          const uint32_t padded = (sp.len + 7u) & ~7u;
          if (heap + padded > (uint32_t)kParamHeap) return OBGPU_NOT_SUPPORTED;
          memcpy(p.param_heap + heap, sp.ptr, sp.len);
          heap += padded;
        }
        if ((size_t)src.col < b->col_types.size() && obf::store_class_of(b->col_types[(size_t)src.col]) == 5) {
          // string constant: i64 carries the first min(len, 8) bytes (little endian) for the equality prefilter
          uint64_t pre = 0;
          if (sp.ptr) memcpy(&pre, sp.ptr, std::min<uint32_t>(sp.len, 8u));
          pd.i64 = (int64_t)pre;
        }
        p.params[n_params++] = pd;
        ++kept;
      }
      nd.n_params = (int16_t)kept;
      if (null_param || (src.op == OBGPU_WHITE_OP_IN && kept == 0)) nd.op = OP_FALSE;
      if ((size_t)src.col < b->col_types.size() && obf::store_class_of(b->col_types[(size_t)src.col]) == 5 &&
          (src.op == OBGPU_WHITE_OP_EQ || src.op == OBGPU_WHITE_OP_NE || src.op == OBGPU_WHITE_OP_IN)) {
        // equality on strings: two 64-bit screens over the constants -- which lengths (mod 64) and which first bytes (mod 64) occur --
        // let a dictionary entry skip the constant list with two bit tests (lo / span are otherwise unused on string leaves)
        uint64_t len_mask = 0, b0_mask = 0;
        for (int k = 0; k < kept; ++k) {
          const ParamDev &q = p.params[nd.param_begin + k];
          len_mask |= 1ull << (q.len & 63u);
          if (q.len == 0) b0_mask = ~0ull; else b0_mask |= 1ull << ((uint64_t)q.i64 & 63u);
        }
        nd.lo = len_mask;
        nd.span = b0_mask;
        // hash slots instead of the first-byte screen when the constants are distinct under one of the multipliers
        for (int m = 0; m < kStrEqHashTries && kept >= 1 && kept <= 32 && nd.pad == 0; ++m) {
          uint64_t occ = 0;
          bool clash = false;
          for (int k = 0; k < kept && !clash; ++k) {
            const ParamDev &q = p.params[nd.param_begin + k];
            const uint64_t bit = 1ull << str_eq_slot((uint64_t)q.i64, q.len, m);
            clash = (occ & bit) != 0;
            occ |= bit;
          }
          if (clash) continue;
          std::sort(p.params + nd.param_begin, p.params + nd.param_begin + kept, [m](const ParamDev &x, const ParamDev &y) {
            return str_eq_slot((uint64_t)x.i64, x.len, m) < str_eq_slot((uint64_t)y.i64, y.len, m);
          });
          nd.span = occ;
          nd.pad = (int16_t)(m + 1);
        }
      }
      // integer compares reduce to one unsigned range test on the compare image (cmp_image: the datum's low
      // bytes, sign-extended for signed classes)
      {
        const uint8_t t = (size_t)src.col < b->col_types.size() ? b->col_types[(size_t)src.col] : 0xff;
        const int sc = t == 0xff ? 0 : obf::store_class_of(t);
        if (nd.op != OP_FALSE && (sc == 1 || sc == 2) && src.op <= OBGPU_WHITE_OP_BT) {
          const bool sg = sc == 1;
          const uint64_t MIN = sg ? (uint64_t)INT64_MIN : 0ull, MAX = sg ? (uint64_t)INT64_MAX : ~0ull;
          auto less = [&](uint64_t x, uint64_t y) { return sg ? (int64_t)x < (int64_t)y : x < y; };
          const uint64_t c0 = (uint64_t)p.params[nd.param_begin].i64;
          uint64_t lo = MIN, hi = MAX;
          bool empty = false;
          switch (src.op) {
            case OBGPU_WHITE_OP_EQ: case OBGPU_WHITE_OP_NE: lo = hi = c0; break;
            case OBGPU_WHITE_OP_LE: hi = c0; break;
            case OBGPU_WHITE_OP_LT: if (c0 == MIN) empty = true; else hi = c0 - 1; break;
            case OBGPU_WHITE_OP_GE: lo = c0; break;
            case OBGPU_WHITE_OP_GT: if (c0 == MAX) empty = true; else lo = c0 + 1; break;
            case OBGPU_WHITE_OP_BT: lo = c0; hi = (uint64_t)p.params[nd.param_begin + 1].i64; if (less(hi, lo)) empty = true; break;
            default: break;
          }
          if (empty) {
            nd.op = OP_FALSE;
          } else {
            nd.range_ok = 1;
            nd.negate = src.op == OBGPU_WHITE_OP_NE;
            nd.lo = lo;
            nd.span = hi - lo;
          }
        }
      }
      if (nd.op != OP_FALSE && (size_t)src.col < b->col_max_dict.size() && b->col_max_dict[(size_t)src.col] > 0) {
        if (p.n_slots >= 127) return OBGPU_NOT_SUPPORTED;
        nd.slot = (int8_t)p.n_slots++;
        p.bitset_words = std::max<int32_t>(p.bitset_words, (int32_t)((b->col_max_dict[(size_t)src.col] + 31) / 32));
      }
      ++depth;
    } else if (src.kind == OBGPU_NODE_AND || src.kind == OBGPU_NODE_OR) {
      if (src.n_children < 2 || src.n_children > 31 || src.n_children > depth) return OBGPU_INVALID_ARGUMENT;
      nd.n_children = (int16_t)src.n_children;
      depth -= src.n_children - 1;
    } else {
      return OBGPU_INVALID_ARGUMENT;
    }
    if (depth > 31) return OBGPU_NOT_SUPPORTED;
    p.nodes[p.n_nodes++] = nd;
  }
  if (depth != 1) return OBGPU_INVALID_ARGUMENT;
  if (p.n_nodes == 1) p.simple_shape = 1;  // single leaf == AND over one leaf
  if (p.n_nodes >= 3) {
    const FilterNodeDev &root = p.nodes[p.n_nodes - 1];
    bool leaves = root.kind != NODE_WHITE && root.n_children == p.n_nodes - 1;
    for (int i = 0; leaves && i < p.n_nodes - 1; ++i) leaves = p.nodes[i].kind == NODE_WHITE;
    if (leaves) p.simple_shape = root.kind == NODE_AND ? 1 : 2;
  }
  // AND over leaves: range tests on the same column collapse into one (a SQL BETWEEN arrives as >= and <=
  // leaves under an AND node, sql/engine/basic/ob_pushdown_filter.cpp:212-262). Same rows selected.
  if (p.simple_shape == 1 && p.n_nodes >= 3) {
    int n_leaves = p.n_nodes - 1;
    for (int i = 0; i < n_leaves; ++i) {
      FilterNodeDev &a = p.nodes[i];
      if (!a.range_ok || a.negate || a.op == OP_FALSE) continue;
      const uint8_t t = (size_t)p.used_col[a.used_idx] < b->col_types.size() ? b->col_types[(size_t)p.used_col[a.used_idx]] : 0xff;
      const bool sg = t != 0xff && obf::store_class_of(t) == 1;
      auto less = [&](uint64_t x, uint64_t y) { return sg ? (int64_t)x < (int64_t)y : x < y; };
      for (int j = i + 1; j < n_leaves;) {
        const FilterNodeDev &c = p.nodes[j];
        if (c.used_idx != a.used_idx || !c.range_ok || c.negate || c.op == OP_FALSE) { ++j; continue; }
        uint64_t lo = a.lo, hi = a.lo + a.span;
        const uint64_t clo = c.lo, chi = c.lo + c.span;
        if (less(lo, clo)) lo = clo;
        if (less(chi, hi)) hi = chi;
        if (less(hi, lo)) { a.op = OP_FALSE; a.range_ok = 0; }
        else { a.lo = lo; a.span = hi - lo; a.op = OP_BT; }  // op is informational once range_ok is set
        for (int k = j; k + 1 < p.n_nodes; ++k) p.nodes[k] = p.nodes[k + 1];
        --p.n_nodes;
        --n_leaves;
        if (a.op == OP_FALSE) break;
      }
    }
    if (n_leaves == 1) p.n_nodes = 1;            // a single leaf needs no AND node
    else p.nodes[p.n_nodes - 1].n_children = (int16_t)n_leaves;
  }
  return OBGPU_SUCCESS;
}

// run-table slots for used columns that are RLE-coded in some block
static void assign_rle_slots(const obgpu_batch *b, ScanParams &p) {
  p.n_rle_slots = 0;
  p.rle_runs_cap = 0;
  for (int i = 0; i < kMaxUsedCols; ++i) p.used_rle_slot[i] = -1;
  for (int i = 0; i < p.n_used; ++i) {
    const size_t col = (size_t)p.used_col[i];
    if (col < b->col_max_rle.size() && b->col_max_rle[col] > 0) {
      p.used_rle_slot[i] = (int8_t)p.n_rle_slots++;
      p.rle_runs_cap = std::max<int32_t>(p.rle_runs_cap, (int32_t)std::min<uint32_t>(b->col_max_rle[col], 65535u));
    }
  }
  const uint32_t rows_cap = std::max<uint32_t>(b->max_rows, 32u);
  p.rows_cap = rows_cap;
  p.words_cap = (rows_cap + 31u) / 32u;
  p.rle_slot_bytes = p.n_rle_slots > 0 ? ((p.words_cap * 6u + 15u) & ~15u) : 0u;
}

// single-block kernels: [block][bitsets][rle tables][descs]
static void layout_smem(const obgpu_batch *b, ScanParams &p, bool /*need_sel*/) {
  assign_rle_slots(b, p);
  uint32_t off = (b->max_block_bytes + 16u + 127u) & ~127u;
  p.smem_bitset = off; off += ((uint32_t)p.n_slots * (uint32_t)p.bitset_words * 4u + 15u) & ~15u;
  p.smem_rle = off;   off += (uint32_t)p.n_rle_slots * p.rle_slot_bytes;
  p.smem_desc = off;  off += (uint32_t)sizeof(ColDesc) * (uint32_t)std::max(p.n_used, 1);
  p.smem_total = (off + 15u) & ~15u;
}

// project kernel: [staged block or packed column regions][bitsets][scratch = sel|bm|wpre|per-warp rle|plans];
// count kernel: per warp descs | bm | bitsets | staging buffer
static void layout_smem_scan(const obgpu_batch *b, ScanParams &p, int max_smem) {
  assign_rle_slots(b, p);
  p.no_stage = 0;
  p.stage_bytes = (b->max_block_bytes + 16u + 127u) & ~127u;
  {
    // stage only the projected columns when that is clearly less than the whole block (upper bound:
    // per-column maximum region over the batch's blocks)
    uint64_t sum = 0;
    bool known = p.n_proj > 0;
    for (int i = 0; i < p.n_proj && known; ++i) {
      const size_t col = (size_t)p.used_col[p.proj_used[i]];
      if (col >= b->col_span.size() || b->col_span[col] == 0xffffffffu) known = false;   // no single region (CS string bytes)
      else sum += b->col_span[col];
    }
    p.compact = 0;
    if (known && sum * 4 <= (uint64_t)p.stage_bytes * 3) {
      p.compact = 1;
      p.stage_bytes = ((uint32_t)sum + 127u) & ~127u;
    }
    if (const char *e = getenv("OBGPU_PROJECT_COMPACT")) {  // testing knob: force either mode
      const int want = atoi(e);
      if (want == 0) { p.compact = 0; p.stage_bytes = (b->max_block_bytes + 16u + 127u) & ~127u; }
      else if (known && want == 1) { p.compact = 1; p.stage_bytes = ((uint32_t)sum + 127u) & ~127u; }
    }
  }
  uint32_t off = p.stage_bytes;
  p.smem_bitset = off; off += ((uint32_t)p.n_slots * (uint32_t)p.bitset_words * 4u + 15u) & ~15u;
  uint32_t s = 0;
  p.off_sel = s;  s += (p.rows_cap * 2u + 15u) & ~15u;
  p.off_bm = s;   s += (p.words_cap * 4u + 15u) & ~15u;
  p.off_wpre = s; s += (p.words_cap * 4u + 15u) & ~15u;
  p.off_rle = s;
  p.pw_rvals = 0;
  p.pw_rle = p.pw_rvals + (p.n_rle_slots > 0 ? (((uint32_t)p.rle_runs_cap + 2u) * 8u) : 0u);
  p.pw_bytes = (p.pw_rle + (p.n_rle_slots > 0 ? p.words_cap * 6u : 0u) + 15u) & ~15u;
  p.off_desc = s; s += p.pw_bytes * (uint32_t)kWarps;
  p.off_plans = s; s += (uint32_t)sizeof(ColDesc) * (uint32_t)std::max(p.n_proj, 1);
  p.scratch_bytes = (s + 127u) & ~127u;
  p.smem_scratch = (off + 127u) & ~127u;
  p.smem_total = p.smem_scratch + p.scratch_bytes;
  if ((int)p.smem_total > max_smem && p.stage_bytes > 0) {
    // the blocks (or the projected column regions) do not fit next to the scratch: no staging at all, and
    // no per-warp run tables either (the global path looks runs up by binary search)
    p.no_stage = 1;
    p.compact = 0;
    p.stage_bytes = 0;
    p.smem_bitset = 0;
    p.pw_rle = p.pw_bytes = 0;
    uint32_t s2 = p.off_desc;          // sel | bm | wpre stay where they are
    p.off_plans = s2; s2 += (uint32_t)sizeof(ColDesc) * (uint32_t)std::max(p.n_proj, 1);
    p.scratch_bytes = (s2 + 127u) & ~127u;
    p.smem_scratch = ((((uint32_t)p.n_slots * (uint32_t)p.bitset_words * 4u + 15u) & ~15u) + 127u) & ~127u;
    p.smem_total = p.smem_scratch + p.scratch_bytes;
  }
  // count kernel, per warp: descs | bm | bitsets
  uint32_t w = 0;
  p.cw_desc = w;   w += ((uint32_t)sizeof(ColDesc) * (uint32_t)std::max(p.n_used, 1) + 15u) & ~15u;
  p.cw_bm = w;     w += (p.words_cap * 4u + 15u) & ~15u;
  p.cw_bitset = w; w += ((uint32_t)p.n_slots * (uint32_t)p.bitset_words * 4u + 15u) & ~15u;
  // staging buffer for one filter column's region at a time (coalesced 16-byte loads); a column whose
  // region exceeds the per-warp budget is read from global memory directly
  uint32_t span = 0;
  for (int i = 0; i < p.n_used; ++i) {
    if (!p.used_in_filter[i] || (size_t)p.used_col[i] >= b->col_span.size()) continue;
    const uint32_t sp = b->col_span[(size_t)p.used_col[i]];
    if (sp <= 24576u) span = std::max(span, sp);  // larger columns are read from global memory
  }
  p.cw_stage_bytes = span;
  p.cw_stage = (w + 15u) & ~15u; w = p.cw_stage + p.cw_stage_bytes;
  p.cw_bytes = (w + 127u) & ~127u;
}


// Small-block pipelined kernels (scan_small.cuh): which of them this scan can use, and their per-warp layouts.
static void layout_pipe(const obgpu_batch *b, ScanParams &p, int max_smem) {
  p.pipe_count = p.pipe_project = 0;
  bool want = b->max_rows <= 512;
  if (const char *e = getenv("OBGPU_PIPE")) want = atoi(e) != 0;   // testing knob: force the path on / off
  if (!want) return;
  auto r16 = [](uint32_t v) { return (v + 15u) & ~15u; };
  // ---- count: every filter column (= the first pf_n used columns) has a bounded region ----------------------
  if (p.n_nodes > 0 && p.simple_shape != 0) {
    int nf = 0;
    bool ok = true;
    while (nf < p.n_used && p.used_in_filter[nf]) ++nf;
    for (int i = nf; i < p.n_used; ++i) ok = ok && !p.used_in_filter[i];
    ok = ok && nf > 0 && nf <= 8;
    uint32_t off = 0;
    for (int i = 0; i < nf && ok; ++i) {
      const size_t col = (size_t)p.used_col[i];
      const uint32_t sp = col < b->col_span.size() ? b->col_span[col] : 0xffffffffu;
      if (sp == 0xffffffffu || sp > 12288u) { ok = false; break; }
      p.pf_off[i] = off;
      p.pf_span[i] = r16(sp);
      off += r16(sp);
    }
    if (ok) {
      p.pf_n = nf;
      p.pc_meta_bytes = 64u + (uint32_t)nf * (uint32_t)sizeof(ColDesc);
      p.pc_region_bytes = 64u + off;   // kCountHdrBytes
      uint32_t w = 0;
      p.pc_meta = w;   w += 3u * p.pc_meta_bytes;
      p.pc_region = w; w += 2u * p.pc_region_bytes;
      p.pc_bm = w;     w += r16(std::max(p.words_cap, 32u) * 4u) + r16(p.rows_cap * 2u);   // spilled bitmap + survivor list
      p.pc_bitset = w; w += r16((uint32_t)p.n_slots * (uint32_t)p.bitset_words * 4u);
      p.pc_bar = w;    w += 16u;
      p.pc_bytes = ((w + 127u) & ~127u) + 128u;   // slack: ragged tail words read a few refs past the staged region
      if (p.pc_bytes * (uint32_t)kWarps * 2u <= (uint32_t)max_smem) p.pipe_count = 1;   // at least two CTAs per SM
    }
  }
  // ---- project ------------------------------------------------------------------------------------------------------
  if (p.n_proj + p.want_row_ids > 0) {
    bool ok = p.n_proj <= 32;   // one lane per projected column computes and issues its byte ranges
    uint32_t off = 0;
    for (int i = 0; i < p.n_proj && ok; ++i) {
      const size_t col = (size_t)p.used_col[p.proj_used[i]];
      const uint32_t sp = col < b->col_pspan.size() ? b->col_pspan[col] : 0xffffffffu;
      if (sp == 0xffffffffu || sp > 16384u) { ok = false; break; }
      p.pp_off[i] = off;
      p.pp_span[i] = r16(sp);
      off += r16(sp);
    }
    if (ok) {
      p.pp_meta_bytes = 64u + (uint32_t)std::max(p.n_proj, 1) * (uint32_t)sizeof(ColDesc);
      p.pp_list = 0;
      p.pp_hdr_bytes = r16((2u * (uint32_t)kMaxProj + 1u) * 4u);   // deltas + flags
      p.pp_bm_bytes = r16(p.words_cap * 4u);
      p.pp_region_bytes = p.pp_hdr_bytes + p.pp_bm_bytes + off;
      // warp-private RLE scratch: [run values][run table] (same shape as the CTA kernel's)
      p.pw_rvals = 0;
      p.pw_rle = p.n_rle_slots > 0 ? (((uint32_t)p.rle_runs_cap + 2u) * 8u) : 0u;
      p.pw_bytes = r16(p.pw_rle + (p.n_rle_slots > 0 ? p.words_cap * 6u : 0u));
      uint32_t w = 0;
      p.pp_meta = w;   w += 3u * p.pp_meta_bytes;
      p.pp_region = w; w += 2u * p.pp_region_bytes;
      p.pp_sel = w;    w += r16(p.rows_cap * 2u);
      p.pp_wscr = w;   w += p.pw_bytes;
      p.pp_bar = w;    w += 16u;
      p.pp_bytes = (w + 127u) & ~127u;
      if (p.pp_bytes * (uint32_t)kWarps * 2u <= (uint32_t)max_smem) p.pipe_project = 1;
    }
  }
}

// ---- pushed-down aggregates over the dense projected columns ------------------------------------------
struct AggAcc {
  unsigned long long lo, hi;   // SUM: 128-bit; MIN / MAX: lo = value, hi = seen; COUNT: lo
};
__device__ __forceinline__ void add128(unsigned long long &lo, unsigned long long &hi, unsigned long long alo,
                                       unsigned long long ahi) {
  const unsigned long long nlo = lo + alo;
  hi += ahi + (nlo < lo ? 1ull : 0ull);
  lo = nlo;
}
template <typename T>
__device__ __forceinline__ long long agg_load(const void *data, int64_t i, bool sgn) {
  const T v = reinterpret_cast<const T *>(data)[i];
  return sgn ? (long long)(typename std::make_signed<T>::type)v : (long long)(unsigned long long)v;
}
__device__ __forceinline__ long long agg_value(const void *data, int elem_len, bool sgn, int64_t i) {
  if (elem_len == 8) return (long long)reinterpret_cast<const unsigned long long *>(data)[i];
  if (elem_len == 4) return agg_load<uint32_t>(data, i, sgn);
  return agg_load<uint8_t>(data, i, sgn);
}
__global__ void __launch_bounds__(256) obgpu_aggregate_kernel(int kind, const void *a, const uint32_t *a_nulls, int a_len, int a_sgn,
                                                              const void *b, const uint32_t *b_nulls, int b_len, int b_sgn,
                                                              const int64_t *n_rows_ptr, unsigned long long *out) {
  __shared__ unsigned long long s_lo[8], s_hi[8];
  const int64_t n = *n_rows_ptr;
  unsigned long long lo = 0, hi = 0;
  const bool is_min = kind == OBGPU_AGG_MIN, is_max = kind == OBGPU_AGG_MAX;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if ((a_nulls[i >> 5] >> (i & 31)) & 1u) continue;
    if (kind == OBGPU_AGG_SUM_PRODUCT && ((b_nulls[i >> 5] >> (i & 31)) & 1u)) continue;
    const long long va = agg_value(a, a_len, a_sgn != 0, i);
    if (kind == OBGPU_AGG_COUNT) { ++lo; continue; }
    if (kind == OBGPU_AGG_SUM) {
      // 8-byte unsigned columns are zero-extended, everything else sign-extended into 128 bits
      const bool neg = (a_sgn || a_len < 8) ? va < 0 : false;
      add128(lo, hi, (unsigned long long)va, neg ? ~0ull : 0ull);
      continue;
    }
    if (kind == OBGPU_AGG_SUM_PRODUCT) {
      const long long vb = agg_value(b, b_len, b_sgn != 0, i);
      const __int128 pa = (a_sgn || a_len < 8) ? (__int128)va : (__int128)(unsigned long long)va;
      const __int128 pb = (b_sgn || b_len < 8) ? (__int128)vb : (__int128)(unsigned long long)vb;
      const unsigned __int128 pr = (unsigned __int128)(pa * pb);
      add128(lo, hi, (unsigned long long)pr, (unsigned long long)(pr >> 64));
      continue;
    }
    // MIN / MAX in the column's own order
    bool better;
    if (!hi) better = true;
    else if (a_sgn || a_len < 8) better = is_min ? va < (long long)lo : va > (long long)lo;
    else better = is_min ? (unsigned long long)va < lo : (unsigned long long)va > lo;
    if (better) { lo = (unsigned long long)va; hi = 1; }
  }
  // block reduction, then one atomic merge per CTA
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long olo = __shfl_xor_sync(0xffffffffu, lo, o), ohi = __shfl_xor_sync(0xffffffffu, hi, o);
    if (is_min || is_max) {
      bool take = false;
      if (ohi) {
        if (!hi) take = true;
        else if (a_sgn || a_len < 8) take = is_min ? (long long)olo < (long long)lo : (long long)olo > (long long)lo;
        else take = is_min ? olo < lo : olo > lo;
      }
      if (take) { lo = olo; hi = 1; }
    } else {
      add128(lo, hi, olo, ohi);
    }
  }
  if (lane == 0) { s_lo[warp] = lo; s_hi[warp] = hi; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) {
      if (is_min || is_max) {
        bool take = false;
        if (s_hi[w]) {
          if (!hi) take = true;
          else if (a_sgn || a_len < 8) take = is_min ? (long long)s_lo[w] < (long long)lo : (long long)s_lo[w] > (long long)lo;
          else take = is_min ? s_lo[w] < lo : s_lo[w] > lo;
        }
        if (take) { lo = s_lo[w]; hi = 1; }
      } else {
        add128(lo, hi, s_lo[w], s_hi[w]);
      }
    }
    if (is_min || is_max) {
      if (hi) {  // out[0]: order-preserving unsigned key (sign bit flipped for signed columns), out[1]: seen
        const unsigned long long key = (a_sgn || a_len < 8) ? lo ^ (1ull << 63) : lo;
        if (is_min) atomicMin(&out[0], key); else atomicMax(&out[0], key);
        atomicOr(&out[1], 1ull);
      }
    } else {
      const unsigned long long prev = atomicAdd(&out[0], lo);
      atomicAdd(&out[1], hi + ((prev + lo) < prev ? 1ull : 0ull));
    }
  }
}

// Dense result column -> ObDatum[] (12 packed bytes: ptr, {len:29, flag:2, null:1}) + 8-byte value slots for integers.
__global__ void __launch_bounds__(256) obgpu_format_datums_kernel(const void *data, const int32_t *lens, const uint32_t *nulls, int elem_len,
                                                                  int is_string, int64_t row_begin, int64_t n, uint64_t slot_base,
                                                                  uint32_t *out12, uint64_t *slots) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int64_t i = row_begin + k;
  const bool is_null = (nulls[i >> 5] >> (i & 31)) & 1u;
  uint64_t ptr;
  uint32_t pack;
  if (is_string) {
    ptr = is_null ? 0ull : reinterpret_cast<const uint64_t *>(data)[i];
    pack = is_null ? 0x80000000u : ((uint32_t)lens[i] & 0x1fffffffu);
  } else {
    uint64_t v = 0;
    if (!is_null) {
      if (elem_len == 8) v = reinterpret_cast<const uint64_t *>(data)[i];
      else if (elem_len == 4) v = reinterpret_cast<const uint32_t *>(data)[i];
      else v = reinterpret_cast<const uint8_t *>(data)[i];
    }
    slots[k] = v;
    ptr = slot_base + 8ull * (uint64_t)k;
    pack = is_null ? 0x80000000u : (uint32_t)elem_len;
  }
  out12[3 * k] = (uint32_t)ptr;
  out12[3 * k + 1] = (uint32_t)(ptr >> 32);
  out12[3 * k + 2] = pack;
}

struct TempDevResult {
  obgpu_ctx *ctx;
  void *p = nullptr;
  explicit TempDevResult(obgpu_ctx *c) : ctx(c) {}
  cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 16, ctx->stream); }
  ~TempDevResult() { if (p) cudaFreeAsync(p, ctx->stream); }
};

static int check_status(obgpu_ctx *ctx, int status) {
  if (status & ST_CORRUPT) { ctx->err = "corrupt micro block seen on device"; return OBGPU_INVALID_DATA; }
  if (status & ST_UNSUPPORTED) { ctx->err = "column encoding / type not handled by the device path"; return OBGPU_NOT_SUPPORTED; }
  if (status & ST_OVERFLOW) { ctx->err = "result capacity exceeded"; return OBGPU_BUF_NOT_ENOUGH; }
  return OBGPU_SUCCESS;
}

// ---- ObCGBitmap: the selection of a row range shared by the column groups of a table ------------------------------------------
struct obgpu_cg_bitmap {
  obgpu_ctx *ctx = nullptr;
  uint32_t *d_words = nullptr;   // bit r of the range at word r / 32, LSB first; 2 words of slack behind the last one
  int64_t n_rows = 0;
};

// 32 bits of a bit array starting at an arbitrary bit position
__device__ __forceinline__ uint32_t bits_at(const uint32_t *__restrict__ w, int64_t bit) {
  const int64_t i = bit >> 5;
  const uint32_t sh = (uint32_t)(bit & 31);
  return __funnelshift_r(w[i], w[i + 1], sh);
}

// One warp per block: the block's rows in the range bitmap -> its packed selection words + selected count (what the count kernel
// produces from a filter)
__global__ void __launch_bounds__(128) obgpu_bitmap_slice_kernel(const uint32_t *__restrict__ cg_words, int64_t cg_rows, int64_t row_offset,
                                                                 const int64_t *__restrict__ row_start, const uint32_t *__restrict__ rows,
                                                                 const int64_t *__restrict__ bm_word_off, int n_blocks,
                                                                 uint32_t *__restrict__ bitmap_words, uint32_t *__restrict__ counts) {
  const int blk = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (blk >= n_blocks) return;
  const uint32_t n = rows[blk];
  const int64_t g0 = row_offset + row_start[blk];
  uint32_t cnt = 0;
  for (uint32_t w = (uint32_t)lane; w < (n + 31u) / 32u; w += 32u) {
    const int64_t g = g0 + 32ll * w;
    uint32_t v = (g >= 0 && g < cg_rows) ? bits_at(cg_words, g) : 0u;
    const uint32_t valid = n - 32u * w >= 32u ? 0xffffffffu : ((1u << (n - 32u * w)) - 1u);
    v &= valid;
    if (g + 32 > cg_rows && g < cg_rows) v &= (uint32_t)((1ull << (cg_rows - g)) - 1ull);
    bitmap_words[bm_word_off[blk] + w] = v;
    cnt += __popc(v);
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) counts[blk] = cnt;
}

static int scan_common(obgpu_batch *b, const obgpu_scan_spec *spec, const obgpu_cg_bitmap *ext_bm, int64_t ext_row_offset, obgpu_result **out);

extern "C" {

int obgpu_scan(obgpu_batch *b, const obgpu_scan_spec *spec, obgpu_result **out) { return scan_common(b, spec, nullptr, 0, out); }

}  // extern "C"

static int scan_common(obgpu_batch *b, const obgpu_scan_spec *spec, const obgpu_cg_bitmap *ext_bm, int64_t ext_row_offset, obgpu_result **out) {
  if (!b || !spec || !out) return OBGPU_INVALID_ARGUMENT;
  if (ext_bm && spec->filter && spec->filter->n_nodes > 0) return OBGPU_INVALID_ARGUMENT;   // the bitmap IS the selection
  obgpu_ctx *ctx = b->ctx;
  if (spec->n_proj < 0 || spec->n_proj > kMaxProj || (spec->n_proj > 0 && !spec->proj_cols))
    return spec->n_proj > kMaxProj ? OBGPU_NOT_SUPPORTED : OBGPU_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  ScanParams p;
  memset(&p, 0, sizeof(p));
  int ret = build_filter(ctx, b, spec->filter, p);
  if (ret != OBGPU_SUCCESS) return ret;
  obgpu_result *r = new (std::nothrow) obgpu_result();
  if (!r) return OBGPU_ALLOCATE_MEMORY_FAILED;
  r->batch = b;
  r->ctx = ctx;
  r->n_proj = spec->n_proj;
  r->cap = spec->max_selected_rows > 0 ? std::min<int64_t>(spec->max_selected_rows, b->total_rows) : b->total_rows;
  // column types were captured at open time (an SSTable has one schema; 0xff = blocks disagree)
  for (int c = 0; c < spec->n_proj; ++c) {
    const int32_t col = spec->proj_cols[c];
    if (col < 0 || (uint32_t)col >= b->max_cols) { delete r; return OBGPU_INVALID_ARGUMENT; }
    const int ui = used_index(p, col);
    if (ui < 0) { delete r; return OBGPU_NOT_SUPPORTED; }
    p.used_in_proj[ui] = 1;
    p.proj_used[c] = (int16_t)ui;
  }
  p.n_proj = spec->n_proj;
  p.want_row_ids = spec->want_row_ids ? 1 : 0;
  p.string_base = spec->string_base;
  r->string_base = spec->string_base;
  // the caller's selectivity estimate (max_selected_rows): when it says at most 1/16 of the rows survive, most
  // blocks will be sparse and the warp-per-block kernel takes them
  const bool selects = p.n_nodes > 0 || ext_bm != nullptr;   // some rows may be dropped: bitmap words + counts exist
  p.sparse_split = (selects && r->cap * 16 <= b->total_rows) ? 1 : 0;
  if (const char *e = getenv("OBGPU_SPARSE_SPLIT")) p.sparse_split = atoi(e) ? (selects ? 1 : 0) : 0;  // testing knob
  layout_smem_scan(b, p, ctx->max_smem_optin);
  layout_pipe(b, p, ctx->max_smem_optin);
  if ((int)p.smem_total > ctx->max_smem_optin && !p.pipe_project) {
    ctx->err = "scan working set exceeds shared memory";
    delete r;
    return OBGPU_NOT_SUPPORTED;
  }
  // ---- result arena: [zeroed region | data] ---------------------------------------------------------
  const int32_t n = b->n_blocks;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
  const size_t o_misc = take(256 + kMaxProj * 4);  // status, has_null
  size_t o_nulls[kMaxProj];
  const size_t null_bytes = (size_t)((r->cap + 63) / 64) * 8;
  for (int c = 0; c < spec->n_proj; ++c) o_nulls[c] = take(null_bytes);
  const size_t zero_bytes = off;
  const size_t o_counts = take((size_t)n * 4);
  const size_t o_chunk = take(((size_t)n / kPrefixChunk + 2) * 8);
  const size_t o_sel = take(((size_t)n + 1) * 8);
  const size_t o_bm = take((size_t)b->bm_word_off[(size_t)n] * 4 + 4);
  const size_t o_rid = spec->want_row_ids ? take((size_t)r->cap * 4) : 0;
  const bool use_skip = b->d_agg != nullptr && p.n_nodes > 0;
  const size_t o_blk_const = use_skip ? take((size_t)n) : 0;
  const size_t o_leaf_const = use_skip ? take((size_t)n * (size_t)p.n_nodes) : 0;
  size_t o_data[kMaxProj], o_lens[kMaxProj];
  for (int c = 0; c < spec->n_proj; ++c) {
    const int t = b->col_types[(size_t)spec->proj_cols[c]];
    o_data[c] = 0;
    o_lens[c] = 0;
    const int sc = obf::store_class_of((uint8_t)t);
    if (sc == 0) { ctx->err = "projected column type not handled by the device path"; delete r; return OBGPU_NOT_SUPPORTED; }
    r->cols[c].obj_type = t;
    r->cols[c].is_string = sc == 5;
    r->cols[c].elem_len = sc == 5 ? 8 : obf::datum_len_of((uint8_t)t);
    o_data[c] = take((size_t)r->cap * (size_t)r->cols[c].elem_len);
    if (sc == 5) o_lens[c] = take((size_t)r->cap * 4);
  }
  r->arena_bytes = off;
  cudaError_t e = cudaMallocAsync(&r->arena, r->arena_bytes, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); delete r; return OBGPU_ALLOCATE_MEMORY_FAILED; }
  uint8_t *a = (uint8_t *)r->arena;
  e = cudaMemsetAsync(a, 0, zero_bytes, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); obgpu_result_free(r); return OBGPU_ERR_SYS; }
  p.image = b->d_image;
  p.blk_off = b->d_blk_off;
  p.blk_size = b->d_blk_size;
  p.bm_word_off = b->d_bm_word_off;
  p.n_blocks = n;
  p.plans = b->d_plans;
  p.rows = b->d_rows;
  p.recs = b->d_recs;
  p.xf = reinterpret_cast<const XformRecFwd *>(b->d_xf);
  p.max_cols = (int32_t)b->max_cols;
  p.counts = (uint32_t *)(a + o_counts);
  p.status = (int32_t *)(a + o_misc + 64);
  p.has_null = (int32_t *)(a + o_misc + 128);
  p.sel_offset = (int64_t *)(a + o_sel);
  p.bitmap_words = (uint32_t *)(a + o_bm);
  p.row_ids = spec->want_row_ids ? (int32_t *)(a + o_rid) : nullptr;
  p.out_cap = r->cap;
  for (int c = 0; c < spec->n_proj; ++c) {
    r->cols[c].data = a + o_data[c];
    r->cols[c].lens = r->cols[c].is_string ? (int32_t *)(a + o_lens[c]) : nullptr;
    r->cols[c].nulls = (uint32_t *)(a + o_nulls[c]);
    p.out_data[c] = r->cols[c].data;
    p.out_lens[c] = r->cols[c].lens;
    p.out_nulls[c] = r->cols[c].nulls;
  }
  r->d_has_null = p.has_null;
  r->d_status = p.status;
  r->d_sel_offset = p.sel_offset;
  r->d_bitmap = p.bitmap_words;
  r->d_row_ids = p.row_ids;
  r->no_filter = !selects;
  r->d_skip_counters = (unsigned long long *)(a + o_misc + 16);
  // ---- launches: [skip index ->] count (filter) -> prefix -> project --------------------------------
  const int pslot = (int)(ctx->prof_count % obgpu_ctx::kProfRing);
  if (ctx->profiling) cudaEventRecord(ctx->ev0[pslot], ctx->stream);
  if (use_skip) {
    skipidx::skip_index_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(p, b->d_agg, b->d_agg_off, a + o_blk_const,
                                                                        a + o_leaf_const, r->d_skip_counters);
    ctx->launches++;
    p.blk_const = a + o_blk_const;
    p.leaf_const = a + o_leaf_const;
  }
  if (ext_bm) {   // ObCGRowScanner::get_next_rows(bitmap): another column group's filter already chose the rows
    obgpu_bitmap_slice_kernel<<<(unsigned)(((int64_t)n * 32 + 127) / 128), 128, 0, ctx->stream>>>(
        ext_bm->d_words, ext_bm->n_rows, ext_row_offset, b->d_row_start, b->d_rows, b->d_bm_word_off, n, p.bitmap_words, p.counts);
    ctx->launches++;
  } else if (p.n_nodes > 0) {
    const uint32_t cw_total = p.cw_bytes * (uint32_t)kWarps;
    if ((int)cw_total > ctx->max_smem_optin) {
      ctx->err = "filter working set exceeds shared memory";
      obgpu_result_free(r);
      return OBGPU_NOT_SUPPORTED;
    }
    if (p.pipe_count) {
      const int smem = (int)(p.pc_bytes * (uint32_t)kWarps);
      int occ = 1;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, obgpu_count_pipe_kernel, kThreads, smem);
      const int grid = std::min((n + kWarps - 1) / kWarps, std::max(1, occ) * ctx->sm_count);
      obgpu_count_pipe_kernel<<<grid, kThreads, smem, ctx->stream>>>(p);
    } else {
      obgpu_count_kernel<<<(n + kWarps - 1) / kWarps, kThreads, cw_total, ctx->stream>>>(p);
    }
    ctx->launches++;
  }
  {
    const int n_chunks = (n + kPrefixChunk - 1) / kPrefixChunk;
    const uint32_t *cnts = selects ? p.counts : b->d_rows;
    obgpu_prefix_local_kernel<<<n_chunks, 256, 0, ctx->stream>>>(cnts, n, p.sel_offset, (unsigned long long *)(a + o_chunk));
    obgpu_prefix_fix_kernel<<<n_chunks + 1, 256, 0, ctx->stream>>>(n, n_chunks, p.sel_offset, (const unsigned long long *)(a + o_chunk));
    ctx->launches += 2;
  }
  if (p.n_proj + p.want_row_ids > 0) {
    p.proj_tiles = p.sparse_split ? 8 : 1;
    if (p.pipe_project) {
      const int smem = (int)(p.pp_bytes * (uint32_t)kWarps);
      int occ = 1;
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, obgpu_project_pipe_kernel, kThreads, smem);
      const int grid = std::min((n + kWarps - 1) / kWarps, std::max(1, occ) * ctx->sm_count);
      obgpu_project_pipe_kernel<<<grid, kThreads, smem, ctx->stream>>>(p);
    } else if (p.sparse_split) obgpu_project_kernel<true><<<(n + p.proj_tiles - 1) / p.proj_tiles, kThreads, p.smem_total, ctx->stream>>>(p);
    else obgpu_project_kernel<false><<<n, kThreads, p.smem_total, ctx->stream>>>(p);
    ctx->launches++;
    if (p.sparse_split && !p.pipe_project) {
      const uint32_t per_warp = (((p.rows_cap / 16u + 32u) * 2u + 15u) & ~15u) + (uint32_t)sizeof(ColDesc);
      obgpu_project_sparse_kernel<<<(n + kWarps - 1) / kWarps, kThreads, per_warp * (uint32_t)kWarps, ctx->stream>>>(p);
      ctx->launches++;
    }
  }
  e = cudaGetLastError();
  if (ctx->profiling) {
    cudaEventRecord(ctx->ev1[pslot], ctx->stream);
    ctx->prof_count++;
  }
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); obgpu_result_free(r); return OBGPU_ERR_SYS; }
  *out = r;
  return OBGPU_SUCCESS;
}

extern "C" {

int obgpu_batch_set_agg_rows(obgpu_batch *b, const void *agg_rows, const int64_t *agg_off) {
  if (!b) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = b->ctx;
  cudaSetDevice(ctx->device);
  if (b->d_agg) { cudaFreeAsync(b->d_agg, ctx->stream); b->d_agg = nullptr; }
  if (b->d_agg_off) { cudaFreeAsync(b->d_agg_off, ctx->stream); b->d_agg_off = nullptr; }
  if (!agg_rows && !agg_off) return OBGPU_SUCCESS;   // detach
  if (!agg_rows || !agg_off) return OBGPU_INVALID_ARGUMENT;
  const int32_t n = b->n_blocks;
  if (agg_off[0] < 0) return OBGPU_INVALID_ARGUMENT;
  for (int32_t i = 0; i < n; ++i)
    if (agg_off[i + 1] < agg_off[i] || agg_off[i + 1] - agg_off[i] > UINT16_MAX) return OBGPU_INVALID_ARGUMENT;
  const int64_t lo = agg_off[0], bytes = agg_off[n] - lo;
  // offsets are rebased to the copied range; the stream-ordered copies read the caller's buffers before returning
  std::vector<int64_t> off((size_t)n + 1);
  for (int32_t i = 0; i <= n; ++i) off[(size_t)i] = agg_off[i] - lo;
  CUDA_TRY(ctx, cudaMallocAsync((void **)&b->d_agg, (size_t)bytes + 16, ctx->stream));
  CUDA_TRY(ctx, cudaMallocAsync((void **)&b->d_agg_off, ((size_t)n + 1) * 8, ctx->stream));
  if (bytes > 0)
    CUDA_TRY(ctx, cudaMemcpyAsync(b->d_agg, (const uint8_t *)agg_rows + lo, (size_t)bytes, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(b->d_agg_off, off.data(), ((size_t)n + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

int obgpu_batch_skip_index_filter(obgpu_batch *b, const obgpu_filter *filter, uint8_t *block_mask) {
  if (!b || !filter || !block_mask) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = b->ctx;
  cudaSetDevice(ctx->device);
  const int32_t n = b->n_blocks;
  if (!b->d_agg) {  // no aggregate data: every block is uncertain (ObMicroIndexInfo::has_agg_data() false)
    memset(block_mask, OBGPU_BOOL_MASK_UNCERTAIN, (size_t)n);
    return OBGPU_SUCCESS;
  }
  ScanParams p;
  memset(&p, 0, sizeof(p));
  const int ret = build_filter(ctx, b, filter, p);
  if (ret != OBGPU_SUCCESS) return ret;
  if (p.n_nodes == 0) return OBGPU_INVALID_ARGUMENT;
  p.n_blocks = n;
  p.plans = b->d_plans;
  p.rows = b->d_rows;
  p.max_cols = (int32_t)b->max_cols;
  uint8_t *verdicts = nullptr;   // [n block verdicts][n x n_nodes node verdicts]
  CUDA_TRY(ctx, cudaMallocAsync((void **)&verdicts, (size_t)n * (size_t)(1 + p.n_nodes) + 16, ctx->stream));
  skipidx::skip_index_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(p, b->d_agg, b->d_agg_off, verdicts, verdicts + n, nullptr);
  ctx->launches++;
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaMemcpyAsync(block_mask, verdicts, (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
  cudaFreeAsync(verdicts, ctx->stream);
  if (e != cudaSuccess) { ctx->err = cudaGetErrorString(e); return OBGPU_ERR_SYS; }
  return OBGPU_SUCCESS;
}

int obgpu_result_skip_info(obgpu_result *r, int64_t *always_false_blocks, int64_t *always_true_blocks) {
  if (!r) return OBGPU_INVALID_ARGUMENT;
  if (!r->info_valid) {
    obgpu_result_info info;
    const int ret = obgpu_result_info_get(r, &info);
    if (ret != OBGPU_SUCCESS && ret != OBGPU_BUF_NOT_ENOUGH) return ret;
  }
  if (always_false_blocks) *always_false_blocks = r->skip_false;
  if (always_true_blocks) *always_true_blocks = r->skip_true;
  return OBGPU_SUCCESS;
}

void obgpu_result_free(obgpu_result *r) {
  if (!r) return;
  cudaSetDevice(r->ctx->device);
  if (r->arena) cudaFreeAsync(r->arena, r->ctx->stream);
  delete r;
}

int obgpu_result_info_get(obgpu_result *r, obgpu_result_info *info) {
  if (!r || !info) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  if (!r->info_valid) {
    cudaSetDevice(ctx->device);
    int64_t *hp = (int64_t *)ctx->h_pinned;
    int32_t *hs = (int32_t *)(hp + 1);
    int32_t *hn = hs + 1;
    CUDA_TRY(ctx, cudaMemcpyAsync(hp, r->d_sel_offset + r->batch->n_blocks, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(hs, r->d_status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(hn, r->d_has_null, kMaxProj * 4, cudaMemcpyDeviceToHost, ctx->stream));
    unsigned long long *hk = (unsigned long long *)((uint8_t *)ctx->h_pinned + 1024);
    CUDA_TRY(ctx, cudaMemcpyAsync(hk, r->d_skip_counters, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    r->skip_false = (int64_t)hk[0];
    r->skip_true = (int64_t)hk[1];
    r->info.total_rows = r->batch->total_rows;
    r->info.selected_rows = *hp;
    r->info.n_blocks = r->batch->n_blocks;
    r->info.n_proj = r->n_proj;
    r->status = *hs;
    memcpy(r->has_null, hn, sizeof(r->has_null));
    r->info_valid = true;
  }
  *info = r->info;
  return check_status(ctx, r->status);
}

int obgpu_result_col_get(obgpu_result *r, int32_t i, obgpu_result_col *col) {
  if (!r || !col || i < 0 || i >= r->n_proj) return OBGPU_INVALID_ARGUMENT;
  col->data = r->cols[i].data;
  col->aux = r->cols[i].lens;
  col->nulls = (uint64_t *)r->cols[i].nulls;
  col->elem_len = r->cols[i].elem_len;
  col->is_string = r->cols[i].is_string;
  col->has_null = r->info_valid ? r->has_null[i] : 0;
  col->obj_type = r->cols[i].obj_type;
  return OBGPU_SUCCESS;
}

int obgpu_result_block_tables(obgpu_result *r, const int64_t **sel_offset_dev, const uint32_t **bitmap_words_dev,
                              const int64_t **bitmap_word_offset_dev, const int32_t **row_ids_dev) {
  if (!r) return OBGPU_INVALID_ARGUMENT;
  if (sel_offset_dev) *sel_offset_dev = r->d_sel_offset;
  if (bitmap_words_dev) *bitmap_words_dev = r->d_bitmap;
  if (bitmap_word_offset_dev) *bitmap_word_offset_dev = r->batch->d_bm_word_off;
  if (row_ids_dev) *row_ids_dev = r->d_row_ids;
  return OBGPU_SUCCESS;
}

int obgpu_result_aggregate(obgpu_result *r, int32_t kind, int32_t col_a, int32_t col_b, int64_t out[2]) {
  if (!r || !out || kind < OBGPU_AGG_COUNT || kind > OBGPU_AGG_MAX || col_a < 0 || col_a >= r->n_proj) return OBGPU_INVALID_ARGUMENT;
  if (kind == OBGPU_AGG_SUM_PRODUCT && (col_b < 0 || col_b >= r->n_proj)) return OBGPU_INVALID_ARGUMENT;
  const ResultCol &a = r->cols[col_a];
  const ResultCol &b = r->cols[kind == OBGPU_AGG_SUM_PRODUCT ? col_b : col_a];
  if (a.is_string || b.is_string) return OBGPU_NOT_SUPPORTED;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  {
    // the scan's own status first: after a capacity overflow sel_offset[n_blocks] exceeds the arena's row
    // capacity and the dense columns hold gaps -- nothing may be read from them
    obgpu_result_info info;
    const int ret = obgpu_result_info_get(r, &info);
    if (ret != OBGPU_SUCCESS) return ret;
  }
  unsigned long long *d_out = nullptr;
  CUDA_TRY(ctx, cudaMallocAsync((void **)&d_out, 32, ctx->stream));
  CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0, 32, ctx->stream));
  if (kind == OBGPU_AGG_MIN) CUDA_TRY(ctx, cudaMemsetAsync(d_out, 0xff, 8, ctx->stream));
  const int a_sgn = obf::store_class_of((uint8_t)a.obj_type) == 1, b_sgn = obf::store_class_of((uint8_t)b.obj_type) == 1;
  // number of selected rows: last entry of the prefix (device resident: no host round trip before the launch)
  obgpu_aggregate_kernel<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(kind, a.data, a.nulls, a.elem_len, a_sgn, b.data, b.nulls, b.elem_len,
                                                                    b_sgn, r->d_sel_offset + r->batch->n_blocks, d_out);
  ctx->launches++;
  unsigned long long h[2] = {0, 0};
  CUDA_TRY(ctx, cudaMemcpyAsync(h, d_out, 16, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  cudaFreeAsync(d_out, ctx->stream);
  if ((kind == OBGPU_AGG_MIN || kind == OBGPU_AGG_MAX) && (a_sgn || a.elem_len < 8)) h[0] ^= 1ull << 63;
  out[0] = (int64_t)h[0];
  out[1] = (int64_t)h[1];
  return OBGPU_SUCCESS;
}

int obgpu_result_fetch_cols(obgpu_result *r, int32_t n_cols, const int32_t *cols, int64_t row_begin, int64_t row_count,
                            void *const *host_data, void *const *host_aux, uint64_t *const *host_nulls) {
  if (!r || n_cols < 0 || (n_cols > 0 && !cols) || row_begin < 0 || row_count < 0 || row_begin + row_count > r->cap)
    return OBGPU_INVALID_ARGUMENT;
  for (int32_t k = 0; k < n_cols; ++k)
    if (cols[k] < 0 || cols[k] >= r->n_proj) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  if (row_count == 0 || n_cols == 0) return OBGPU_SUCCESS;
  const int64_t w0 = row_begin / 64, w1 = (row_begin + row_count + 63) / 64;
  const int sh = (int)(row_begin % 64);
  std::vector<std::vector<uint64_t>> tmp((size_t)n_cols);
  // every copy is enqueued before the single synchronisation
  for (int32_t k = 0; k < n_cols; ++k) {
    const ResultCol &c = r->cols[cols[k]];
    void *hd = host_data ? host_data[k] : nullptr;
    void *ha = host_aux ? host_aux[k] : nullptr;
    uint64_t *hn = host_nulls ? host_nulls[k] : nullptr;
    if (hd)
      CUDA_TRY(ctx, cudaMemcpyAsync(hd, (uint8_t *)c.data + row_begin * c.elem_len, (size_t)row_count * c.elem_len,
                                    cudaMemcpyDeviceToHost, ctx->stream));
    if (ha && c.lens)
      CUDA_TRY(ctx, cudaMemcpyAsync(ha, c.lens + row_begin, (size_t)row_count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (hn) {
      if (sh == 0) {
        CUDA_TRY(ctx, cudaMemcpyAsync(hn, (uint64_t *)c.nulls + w0, (size_t)(w1 - w0) * 8, cudaMemcpyDeviceToHost, ctx->stream));
      } else {
        tmp[(size_t)k].resize((size_t)(w1 - w0) + 1, 0);
        CUDA_TRY(ctx, cudaMemcpyAsync(tmp[(size_t)k].data(), (uint64_t *)c.nulls + w0, (size_t)(w1 - w0) * 8,
                                      cudaMemcpyDeviceToHost, ctx->stream));
      }
    }
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const int64_t ow = (row_count + 63) / 64;
  for (int32_t k = 0; k < n_cols; ++k) {
    uint64_t *hn = host_nulls ? host_nulls[k] : nullptr;
    if (!hn) continue;
    if (sh != 0) {
      const std::vector<uint64_t> &t = tmp[(size_t)k];
      for (int64_t j = 0; j < ow; ++j) hn[j] = (t[(size_t)j] >> sh) | (t[(size_t)j + 1] << (64 - sh));
    }
    if (row_count % 64) hn[ow - 1] &= (1ull << (row_count % 64)) - 1ull;
  }
  return OBGPU_SUCCESS;
}

int obgpu_result_fetch_col(obgpu_result *r, int32_t i, int64_t row_begin, int64_t row_count, void *host_data,
                           void *host_aux, uint64_t *host_nulls) {
  if (!r || i < 0 || i >= r->n_proj) return OBGPU_INVALID_ARGUMENT;
  void *hd[1] = {host_data}, *ha[1] = {host_aux};
  uint64_t *hn[1] = {host_nulls};
  return obgpu_result_fetch_cols(r, 1, &i, row_begin, row_count, hd, ha, hn);
}

int obgpu_result_fetch_datums(obgpu_result *r, int32_t i, int64_t row_begin, int64_t row_count, obgpu_datum *host_datums,
                              void *host_slots) {
  if (!r || i < 0 || i >= r->n_proj || row_begin < 0 || row_count < 0 || row_begin + row_count > r->cap || !host_datums)
    return OBGPU_INVALID_ARGUMENT;
  const ResultCol &c = r->cols[i];
  if (!c.is_string && !host_slots) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  if (row_count == 0) return OBGPU_SUCCESS;
  TempDevResult tmp(ctx);
  const size_t o_slots = ((size_t)row_count * 12 + 255) & ~(size_t)255;
  CUDA_TRY(ctx, tmp.alloc(o_slots + (c.is_string ? 0 : (size_t)row_count * 8)));
  uint8_t *d12 = (uint8_t *)tmp.p;
  uint64_t *dslots = c.is_string ? nullptr : (uint64_t *)((uint8_t *)tmp.p + o_slots);
  obgpu_format_datums_kernel<<<(unsigned)((row_count + 255) / 256), 256, 0, ctx->stream>>>(
      c.data, c.lens, c.nulls, c.elem_len, c.is_string, row_begin, row_count, (uint64_t)(uintptr_t)host_slots, (uint32_t *)d12, dslots);
  ctx->launches++;
  CUDA_TRY(ctx, cudaGetLastError());
  CUDA_TRY(ctx, cudaMemcpyAsync(host_datums, d12, (size_t)row_count * 12, cudaMemcpyDeviceToHost, ctx->stream));
  if (dslots) CUDA_TRY(ctx, cudaMemcpyAsync(host_slots, dslots, (size_t)row_count * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

int obgpu_result_fetch_sel_offsets(obgpu_result *r, int64_t *host_sel_offset) {
  if (!r || !host_sel_offset) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  CUDA_TRY(ctx, cudaMemcpyAsync(host_sel_offset, r->d_sel_offset, ((size_t)r->batch->n_blocks + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

int obgpu_result_fetch_row_ids(obgpu_result *r, int64_t row_begin, int64_t row_count, int32_t *host_row_ids) {
  if (!r || !host_row_ids || !r->d_row_ids || row_begin < 0 || row_count < 0 || row_begin + row_count > r->cap)
    return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  if (row_count == 0) return OBGPU_SUCCESS;
  CUDA_TRY(ctx, cudaMemcpyAsync(host_row_ids, r->d_row_ids + row_begin, (size_t)row_count * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

int obgpu_result_fetch_bitmap(obgpu_result *r, int32_t block, int64_t start, int64_t count, uint8_t *host_bitmap_bytes) {
  if (!r || !host_bitmap_bytes || block < 0 || block >= r->batch->n_blocks || start < 0 || count < 0 ||
      start + count > (int64_t)r->batch->row_count[(size_t)block])
    return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = r->ctx;
  cudaSetDevice(ctx->device);
  if (r->no_filter) {  // no predicate: every row is selected, the count kernel did not run
    memset(host_bitmap_bytes, 1, (size_t)count);
    return OBGPU_SUCCESS;
  }
  const int64_t w0 = r->batch->bm_word_off[(size_t)block], nw = r->batch->bm_word_off[(size_t)block + 1] - w0;
  std::vector<uint32_t> words((size_t)nw);
  CUDA_TRY(ctx, cudaMemcpyAsync(words.data(), r->d_bitmap + w0, (size_t)nw * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  for (int64_t i = 0; i < count; ++i) {
    const int64_t row = start + i;
    host_bitmap_bytes[i] = (words[(size_t)(row >> 5)] >> (row & 31)) & 1u;
  }
  return OBGPU_SUCCESS;
}

}  // extern "C"

// =================================================================================================
// Reference-granularity entry points (one block, one call). Same device code, one-CTA kernels.
// =================================================================================================
namespace {

struct TempDev {
  obgpu_ctx *ctx;
  void *p = nullptr;
  explicit TempDev(obgpu_ctx *c) : ctx(c) {}
  cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes ? bytes : 16, ctx->stream); }
  ~TempDev() { if (p) cudaFreeAsync(p, ctx->stream); }
};

int run_filter_block(obgpu_batch *b, int32_t block, const obgpu_filter *f, int64_t start, int64_t count,
                     uint8_t *result_bitmap) {
  if (!b || !f || !result_bitmap || block < 0 || block >= b->n_blocks || start < 0 || count < 0 ||
      start + count > (int64_t)b->row_count[(size_t)block])
    return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = b->ctx;
  cudaSetDevice(ctx->device);
  ScanParams p;
  memset(&p, 0, sizeof(p));
  int ret = build_filter(ctx, b, f, p);
  if (ret != OBGPU_SUCCESS) return ret;
  if (p.n_nodes == 0) return OBGPU_INVALID_ARGUMENT;
  if (count == 0) return OBGPU_SUCCESS;
  layout_smem(b, p, false);
  if ((int)p.smem_total > ctx->max_smem_optin) return OBGPU_NOT_SUPPORTED;
  TempDev tmp(ctx);
  CUDA_TRY(ctx, tmp.alloc((size_t)count + 64));
  uint8_t *d_bytes = (uint8_t *)tmp.p + 64;
  CUDA_TRY(ctx, cudaMemsetAsync(tmp.p, 0, 64, ctx->stream));
  p.image = b->d_image;
  p.blk_off = b->d_blk_off;
  p.blk_size = b->d_blk_size;
  p.bm_word_off = b->d_bm_word_off;
  p.n_blocks = b->n_blocks;
  p.status = (int32_t *)tmp.p;
  obgpu_filter_block_kernel<<<1, kThreads, p.smem_total, ctx->stream>>>(p, block, start, count, d_bytes);
  CUDA_TRY(ctx, cudaGetLastError());
  ctx->launches++;
  int32_t *hs = (int32_t *)ctx->h_pinned;
  CUDA_TRY(ctx, cudaMemcpyAsync(hs, tmp.p, 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(result_bitmap, d_bytes, (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return check_status(ctx, *hs);
}

int run_project_block(obgpu_batch *b, int32_t block, int32_t col, const int32_t *row_ids, int64_t row_cap,
                      int64_t vec_offset, uint64_t string_base, void *data, int32_t elem_len, int32_t *lens,
                      uint64_t *nulls, int32_t *has_null, bool want_string) {
  if (!b || !row_ids || !data || block < 0 || block >= b->n_blocks || row_cap < 0 || vec_offset < 0 || col < 0)
    return OBGPU_INVALID_ARGUMENT;
  if (want_string && !lens) return OBGPU_INVALID_ARGUMENT;
  if (!want_string && elem_len != 8 && elem_len != 4 && elem_len != 1) return OBGPU_INVALID_ARGUMENT;
  if (row_cap == 0) return OBGPU_SUCCESS;
  obgpu_ctx *ctx = b->ctx;
  cudaSetDevice(ctx->device);
  ScanParams p;
  memset(&p, 0, sizeof(p));
  p.n_used = 1;
  p.used_col[0] = col;
  layout_smem(b, p, false);
  if ((int)p.smem_total > ctx->max_smem_optin) return OBGPU_NOT_SUPPORTED;
  const size_t el = want_string ? 8 : (size_t)elem_len;
  const int64_t total = vec_offset + row_cap;
  const size_t null_words32 = (size_t)((total + 63) / 64) * 2;
  size_t off = 256;
  const size_t o_rid = off; off += ((size_t)row_cap * 4 + 255) & ~(size_t)255;
  const size_t o_nulls = off; off += (null_words32 * 4 + 255) & ~(size_t)255;
  const size_t o_data = off; off += ((size_t)total * el + 255) & ~(size_t)255;
  const size_t o_lens = off; off += want_string ? (((size_t)total * 4 + 255) & ~(size_t)255) : 0;
  TempDev tmp(ctx);
  CUDA_TRY(ctx, tmp.alloc(off));
  uint8_t *a = (uint8_t *)tmp.p;
  CUDA_TRY(ctx, cudaMemsetAsync(a, 0, o_data, ctx->stream));  // status, has_null, row ids, nulls
  CUDA_TRY(ctx, cudaMemcpyAsync(a + o_rid, row_ids, (size_t)row_cap * 4, cudaMemcpyHostToDevice, ctx->stream));
  // the caller's vector keeps whatever it held in NULL slots / outside the window: seed the device
  // image with it so that the copy back is a pure overlay (reference leaves NULL slots unwritten)
  CUDA_TRY(ctx, cudaMemcpyAsync(a + o_data + (size_t)vec_offset * el, (uint8_t *)data + (size_t)vec_offset * el,
                                (size_t)row_cap * el, cudaMemcpyHostToDevice, ctx->stream));
  if (want_string)
    CUDA_TRY(ctx, cudaMemcpyAsync(a + o_lens + (size_t)vec_offset * 4, lens + vec_offset, (size_t)row_cap * 4,
                                  cudaMemcpyHostToDevice, ctx->stream));
  p.image = b->d_image;
  p.blk_off = b->d_blk_off;
  p.blk_size = b->d_blk_size;
  p.n_blocks = b->n_blocks;
  p.status = (int32_t *)a;
  p.has_null = (int32_t *)(a + 64);
  p.string_base = string_base;
  p.xf = reinterpret_cast<const XformRecFwd *>(b->d_xf);
  obgpu_project_block_kernel<<<1, kThreads, p.smem_total, ctx->stream>>>(
      p, block, (const int32_t *)(a + o_rid), row_cap, vec_offset, a + o_data,
      want_string ? (int32_t *)(a + o_lens) : nullptr, (uint32_t *)(a + o_nulls), (int32_t)el);
  CUDA_TRY(ctx, cudaGetLastError());
  ctx->launches++;
  int32_t *hs = (int32_t *)ctx->h_pinned;
  CUDA_TRY(ctx, cudaMemcpyAsync(hs, a, 128 + 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync((uint8_t *)data + (size_t)vec_offset * el, a + o_data + (size_t)vec_offset * el,
                                (size_t)row_cap * el, cudaMemcpyDeviceToHost, ctx->stream));
  if (want_string)
    CUDA_TRY(ctx, cudaMemcpyAsync(lens + vec_offset, a + o_lens + (size_t)vec_offset * 4, (size_t)row_cap * 4,
                                  cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<uint64_t> hnulls(null_words32 / 2);
  CUDA_TRY(ctx, cudaMemcpyAsync(hnulls.data(), a + o_nulls, null_words32 * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const int st = check_status(ctx, hs[0]);
  if (st != OBGPU_SUCCESS) return st;
  if (nulls)
    for (size_t k = 0; k < hnulls.size(); ++k) nulls[k] |= hnulls[k];  // ObBitVector::set semantics
  if (has_null && hs[16]) *has_null = 1;
  return OBGPU_SUCCESS;
}

}  // namespace

extern "C" {

int obgpu_filter_white(obgpu_batch *batch, int32_t block, int32_t col, int32_t op, const obgpu_filter_param *params,
                       int32_t n_params, int64_t start, int64_t count, uint8_t *result_bitmap) {
  obgpu_filter_node nd{};
  nd.kind = OBGPU_NODE_WHITE;
  nd.op = op;
  nd.col = col;
  nd.param_begin = 0;
  nd.n_params = n_params;
  obgpu_filter f{&nd, 1, params, n_params};
  return run_filter_block(batch, block, &f, start, count, result_bitmap);
}

int obgpu_filter_tree(obgpu_batch *batch, int32_t block, const obgpu_filter *filter, int64_t start, int64_t count,
                      uint8_t *result_bitmap) {
  return run_filter_block(batch, block, filter, start, count, result_bitmap);
}

int obgpu_bitmap_to_row_ids(obgpu_ctx *ctx, const uint8_t *bitmap, int64_t bitmap_size, int64_t *from, int64_t to,
                            int64_t limit, int64_t id_offset, int32_t *row_ids, int64_t *row_count) {
  // argument checks of ObBitmap::get_row_ids (ob_bitmap.cpp:547-552)
  if (!ctx || !bitmap || !from || !row_ids || !row_count) return OBGPU_INVALID_ARGUMENT;
  if (*from < 0 || to > bitmap_size || to < *from || limit <= 0 || *from < id_offset) return OBGPU_INVALID_ARGUMENT;
  cudaSetDevice(ctx->device);
  const int64_t span = to - *from;
  if (span == 0) { *row_count = 0; return OBGPU_SUCCESS; }
  const int64_t out_n = std::min(limit, span);
  TempDev tmp(ctx);
  const size_t o_bytes = 64, o_ids = o_bytes + (((size_t)span + 255) & ~(size_t)255);
  CUDA_TRY(ctx, tmp.alloc(o_ids + (size_t)out_n * 4));
  uint8_t *a = (uint8_t *)tmp.p;
  CUDA_TRY(ctx, cudaMemcpyAsync(a + o_bytes, bitmap + *from, (size_t)span, cudaMemcpyHostToDevice, ctx->stream));
  // device bitmap is re-based to *from: ids are (i + *from) - id_offset
  obgpu_bitmap_row_ids_kernel<<<1, kThreads, 0, ctx->stream>>>(a + o_bytes, 0, span, limit, id_offset - *from,
                                                               (int32_t *)(a + o_ids), (int64_t *)a);
  CUDA_TRY(ctx, cudaGetLastError());
  ctx->launches++;
  int64_t *hc = (int64_t *)ctx->h_pinned;
  CUDA_TRY(ctx, cudaMemcpyAsync(hc, a, 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(row_ids, a + o_ids, (size_t)out_n * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  const int64_t n = *hc;
  *row_count = n;
  if (n >= limit) *from = row_ids[limit - 1] + id_offset + 1;
  else *from = to;
  return OBGPU_SUCCESS;
}

int obgpu_project_fixed(obgpu_batch *batch, int32_t block, int32_t col, const int32_t *row_ids, int64_t row_cap,
                        int64_t vec_offset, void *data, int32_t elem_len, uint64_t *nulls, int32_t *has_null) {
  return run_project_block(batch, block, col, row_ids, row_cap, vec_offset, 0, data, elem_len, nullptr, nulls,
                           has_null, false);
}

int obgpu_project_discrete(obgpu_batch *batch, int32_t block, int32_t col, const int32_t *row_ids, int64_t row_cap,
                           int64_t vec_offset, uint64_t string_base, uint64_t *ptrs, int32_t *lens, uint64_t *nulls,
                           int32_t *has_null) {
  return run_project_block(batch, block, col, row_ids, row_cap, vec_offset, string_base, ptrs, 8, lens, nulls,
                           has_null, true);
}

int obgpu_project_datums(obgpu_batch *batch, int32_t block, int32_t col, const int32_t *row_ids, int64_t row_cap, int64_t datum_offset,
                         uint64_t string_base, obgpu_datum *datums) {
  if (!batch || !datums || row_cap < 0 || datum_offset < 0 || col < 0 || (uint32_t)col >= batch->max_cols) return OBGPU_INVALID_ARGUMENT;
  if (row_cap == 0) return OBGPU_SUCCESS;
  const int sc = obf::store_class_of(batch->col_types[(size_t)col]);
  if (sc == 0) return OBGPU_NOT_SUPPORTED;
  const bool is_str = sc == 5;
  const int el = is_str ? 8 : obf::datum_len_of(batch->col_types[(size_t)col]);
  std::vector<uint64_t> data((size_t)row_cap, 0), nulls((size_t)(row_cap + 63) / 64, 0);
  std::vector<int32_t> lens(is_str ? (size_t)row_cap : 0);
  int32_t has_null = 0;
  const int ret = run_project_block(batch, block, col, row_ids, row_cap, 0, string_base, data.data(), el, is_str ? lens.data() : nullptr,
                                    nulls.data(), &has_null, is_str);
  if (ret != OBGPU_SUCCESS) return ret;
  obgpu_datum *out = datums + datum_offset;
  for (int64_t i = 0; i < row_cap; ++i) {
    if ((nulls[(size_t)i / 64] >> (i % 64)) & 1ull) { out[i].pack = OBGPU_DATUM_NULL_BIT; continue; }   // ObDatum::set_null()
    if (is_str) {
      out[i].ptr = data[(size_t)i];
      out[i].pack = (uint32_t)lens[(size_t)i] & 0x1fffffffu;
    } else {
      // load_data_to_datum: MEMCPY through the datum's own pointer (the caller's reserved slot), then the length
      if (out[i].ptr == 0) return OBGPU_INVALID_ARGUMENT;
      memcpy(reinterpret_cast<void *>((uintptr_t)out[i].ptr), reinterpret_cast<const uint8_t *>(data.data()) + (size_t)i * (size_t)el, (size_t)el);
      out[i].pack = (uint32_t)el;
    }
  }
  return OBGPU_SUCCESS;
}

}  // extern "C"

// ---- ObCGBitmap: range bitmaps shared by the column groups of a table ----------------------------------------------------
#include "macro_blocks.cuh"   // macro blocks (disk format) -> page batch, parsed and re-laid on the device
#include "cg_bitmap.cuh"

// ---- string cells as bytes (dense heap): scan results and the per-block entry ------------------------------------------
#include "result_strings.cuh"

// ---- dictionary surface: distinct values, references, black filter on one dictionary column, GROUP BY ----
#include "dict_ops.cuh"

// ---- major-compaction merge (include/obgpu_compaction.h) -----------------------------------------
#include "../../include/obgpu_compaction.h"
#include "merge_kernels.cuh"
#include "merge_exchange.cuh"
#include "merge_streamed.cuh"
#include "encode_kernels.cuh"   // phase B: merged columns -> SSTable bytes + column checksums
#include "encode_codecs.cuh"    // phase B with DICT / RLE / CONST / INTEGER_BASE_DIFF columns, or the codec chosen per micro-block

// ---- host-buffer scan pipeline (include/obgpu_pipeline.h) ------------------------------------------------
#include "host_pipeline.h"
