// Phase B of the compaction on the device: merged column arrays -> PAX micro-blocks (every column RAW), byte for byte the
// blocks the host writer (sstable_writer.cpp: BlockBuilder::encode_raw / build / finish_header) produces for the same rows,
// plus the column checksums of the rows (K16). One kernel, one CTA per micro-block, input read once, output written once:
//
//   stats   : per column max of the stored value image + NULL count (and, fused, the column checksum of the cells); four
//             columns' loads in flight together, warp reductions through redux.sync
//   plan    : warp 0, one lane per column, lays the block out (ObRawEncoder::traverse width rules, ext bits, column stores back
//             to back by a warp scan) and publishes the aligned block size for the look-back at once
//   pack    : cells -> shared-memory image of the block (ext bits, bit-packed and byte-packed values are all "w bits at bit
//             address b": at most three shared atomicOr per cell); the second read of the cells hits L2
//   crc32c  : payload checksum in parallel -- every thread the raw CRC of an odd-word-stride chunk (slicing by 4, tables in
//             shared memory), shifted to its position by ONE carry-less multiplication with x^(32 * words after it) mod P
//             (host-built table) and XOR-reduced; leading zero words cost nothing with init 0 / no final xor
//   offset  : decoupled look-back over the aligned block sizes (tickets in scheduling order, one 64-bit flag per block), resolved
//             by thread 0 while the other warps pack
//   store   : header + checksums, then ONE bulk copy (TMA, cp.async.bulk shared -> global) of the aligned slot
#pragma once
#include <map>
#include <mutex>

namespace enc {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
constexpr int kMaxCols = 64;
constexpr uint32_t kCrcPoly = 0x82f63b78u;   // CRC-32C (Castagnoli), reflected
constexpr uint32_t kHeaderSize = 64u;        // MICRO_HEADER_FIXED_SIZE

struct ColSpec {
  const int64_t *vals;
  const uint8_t *nulls;
  uint64_t store_mask;     // low type_store_size bytes (ColCtx::uval)
  uint8_t obj_type, byte_only, datum_len, enc;   // enc: OBGPU_ENC_* of the column (codec kernel only)
  uint8_t sc, ts, pad[2];                          // store class (1 signed, 2 unsigned), type_store_size
};

struct Params {
  ColSpec col[kMaxCols];
  int32_t n_cols, rowkey_cnt, n_blocks, want_checksums;
  int64_t total_rows, rows_per_block;
  uint32_t align, slot_cap;          // slot_cap: bytes of the shared-memory block image (multiple of align)
  uint32_t lw_max, pad;              // xpow32 holds (kThreads - 1) * lw_max + 1 entries
  uint8_t *image;
  int64_t *blk_off;                  // [n_blocks]
  uint32_t *blk_size;                // [n_blocks] exact bytes, 0: left to the host writer
  unsigned long long *flags;         // [n_blocks] look-back words: state << 62 | bytes
  unsigned long long *checksums;     // [n_cols]
  unsigned long long *totals;        // [0] image bytes, [1] host blocks
  int32_t *ticket;
  const uint32_t *xpow32;            // x^(32 k) mod P, reflected (x^0 = 0x80000000)
};

__device__ __forceinline__ uint32_t gf2_mulmod(uint32_t a, uint32_t b) {
  uint32_t p = 0;
#pragma unroll 8
  for (int i = 0; i < 32; ++i) {
    p ^= (a & 0x80000000u) ? b : 0u;
    a <<= 1;
    b = (b >> 1) ^ ((b & 1u) ? kCrcPoly : 0u);
  }
  return p;
}

__device__ __forceinline__ uint32_t crc_word(const uint32_t *tab, uint32_t crc, uint32_t w) {
  crc ^= w;
  return tab[768 + (crc & 0xffu)] ^ tab[512 + ((crc >> 8) & 0xffu)] ^ tab[256 + ((crc >> 16) & 0xffu)] ^ tab[crc >> 24];
}
__device__ __forceinline__ uint32_t crc_byte(const uint32_t *tab, uint32_t crc, uint32_t b) {
  return tab[(crc ^ b) & 0xffu] ^ (crc >> 8);
}

// get_packing_size (encoding/ob_encoding_util.cpp:37-73): size in bits when bit packing, else in bytes
__device__ __forceinline__ uint32_t packing_size(uint64_t v, bool enable_bp, bool &bp) {
  const uint32_t bits = v == 0 ? 1u : 64u - (uint32_t)__clzll((long long)v);
  if (!enable_bp) {
    bp = false;
    return v <= 0xffull ? 1u : v <= 0xffffull ? 2u : v <= 0xffffffffull ? 4u : 8u;
  }
  uint32_t size = bits / 8u;
  const uint32_t ext = bits % 8u;
  if (ext == 0) { bp = false; return size; }
  if (8u - ext < size / 2u + 1u) { bp = false; return size + 1u; }
  bp = true;
  return bits;
}

struct ColLayout {
  uint32_t store_off;   // byte offset of the column store inside the block
  uint32_t bits_size;   // bytes of the bit area ([ext bits][bit-packed values])
  uint8_t attr, size, bp, has_null;
};

// ---- pieces shared by the RAW kernel and the codec kernel (encode_codecs.cuh); NT: threads of the CTA -------------------------
// crc tables (slicing by 4): tab[k * 256 + i] = crc of byte i followed by k zero bytes
template <int NT>
__device__ __forceinline__ void build_crc_tables(uint32_t *tab, int tid) {
  for (int i = tid; i < 256; i += NT) {
    uint32_t c = (uint32_t)i;
#pragma unroll
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? kCrcPoly ^ (c >> 1) : c >> 1;
    tab[i] = c;
  }
  __syncthreads();
  for (int i = tid; i < 256; i += NT) {
    uint32_t c = tab[i];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      c = (c >> 8) ^ tab[c & 0xffu];
      tab[k * 256 + i] = c;
    }
  }
}

// Stats (+ column checksums): per warp and column the max of the stored value image and the NULL count, into
// s_wmax / s_wnull [NT / 32][n_cols]; four columns at a time, their loads in flight together.
template <int NT, bool CKSUM>
__device__ __forceinline__ void stats_pass(const Params &p, const uint32_t *tab, int64_t row0, uint32_t nrows, unsigned long long *s_wmax,
                                           uint32_t *s_wnull, int tid, int lane, int warp) {
  const int nc = p.n_cols;
  for (int c0 = 0; c0 < nc; c0 += 4) {
    unsigned long long mx[4] = {0, 0, 0, 0}, sum[4] = {0, 0, 0, 0};
    uint32_t nn[4] = {0, 0, 0, 0};
    // ObDatum::checksum(0) starts with the crc32c of the 4 pack_ bytes {len_:29, flag_:2, null_:1}: two values per column
    uint32_t len_crc[4] = {0, 0, 0, 0};
    const uint32_t null_crc = CKSUM ? crc_word(tab, 0u, 0x80000000u) : 0u;
    if (CKSUM) {
#pragma unroll
      for (int j = 0; j < 4; ++j) len_crc[j] = crc_word(tab, 0u, (uint32_t)p.col[min(c0 + j, nc - 1)].datum_len);
    }
    for (uint32_t r = (uint32_t)tid; r < nrows; r += NT) {
      unsigned long long x[4];
      uint32_t nlb[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = min(c0 + j, nc - 1);   // the tail repeats the last column (its results are dropped below)
        x[j] = (unsigned long long)p.col[c].vals[row0 + r];
        nlb[j] = p.col[c].nulls ? p.col[c].nulls[row0 + r] : 0u;
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const ColSpec &cs = p.col[min(c0 + j, nc - 1)];
        const bool is_null = nlb[j] != 0;
        if (is_null) ++nn[j];
        else mx[j] = max(mx[j], x[j] & cs.store_mask);
        if (CKSUM) {   // ... then the crc of the value bytes
          uint32_t crc = is_null ? null_crc : len_crc[j];
          if (!is_null) {
            if (cs.datum_len == 8) {
              crc = crc_word(tab, crc, (uint32_t)x[j]);
              crc = crc_word(tab, crc, (uint32_t)(x[j] >> 32));
            } else if (cs.datum_len == 4) {
              crc = crc_word(tab, crc, (uint32_t)x[j]);
            } else {
              for (uint32_t k = 0; k < cs.datum_len; ++k) crc = crc_byte(tab, crc, (uint32_t)(x[j] >> (8u * k)) & 0xffu);
            }
          }
          sum[j] += crc;
        }
      }
    }
    // warp reductions through redux.sync (one instruction per 32-bit value): 64-bit max as (high word, then the low words of
    // the lanes that hold it); the checksum sum (< 2^32 * rows per lane) as 16-bit digits that cannot overflow 32 bits
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (c0 + j >= nc) break;
      const uint32_t hi = (uint32_t)(mx[j] >> 32), hmax = __reduce_max_sync(0xffffffffu, hi);
      const uint32_t lmax = __reduce_max_sync(0xffffffffu, hi == hmax ? (uint32_t)mx[j] : 0u);
      const uint32_t nsum = __reduce_add_sync(0xffffffffu, nn[j]);
      unsigned long long tot = 0;
      if (CKSUM) {
#pragma unroll
        for (int d = 0; d < 4; ++d) tot += (unsigned long long)__reduce_add_sync(0xffffffffu, (uint32_t)(sum[j] >> (16 * d)) & 0xffffu) << (16 * d);
      }
      if (lane == 0) {
        s_wmax[warp * nc + c0 + j] = ((unsigned long long)hmax << 32) | lmax;
        s_wnull[warp * nc + c0 + j] = nsum;
        if (CKSUM && tot != 0) atomicAdd(p.checksums + c0 + j, tot);
      }
    }
  }
}

// x (w <= 64 bits) at block bit address b of the zeroed shared-memory image: at most three shared atomicOr
__device__ __forceinline__ void or_bits(uint32_t *img32, uint32_t b, uint32_t w, unsigned long long x) {
  const uint32_t sh = b & 31u;
  const unsigned long long xm = w >= 64u ? x : (x & ((1ull << w) - 1ull));
  uint32_t *q = img32 + (b >> 5);
  atomicOr(q, (uint32_t)(xm << sh));
  if (sh + w > 32u) atomicOr(q + 1, (uint32_t)(xm >> (32u - sh)));
  if (sh + w > 64u) atomicOr(q + 2, (uint32_t)(xm >> (64u - sh)));
}

// Output offset (thread 0): decoupled look-back over the aligned sizes (flag word: bits 63..62 state -- 1 aggregate, 2 inclusive
// prefix --, low 62 bits bytes). Tickets are handed out in scheduling order, so every predecessor is running or done.
__device__ __forceinline__ long long look_back(const Params &p, int blk, uint32_t size, uint32_t slot, bool host) {
  volatile unsigned long long *flags = p.flags;
  unsigned long long excl = 0;
  if (blk > 0) {
    int j = blk - 1;
    for (;;) {
      unsigned long long f;
      do { f = flags[j]; } while ((f >> 62) == 0ull);
      excl += f & ((1ull << 62) - 1ull);
      if ((f >> 62) == 2ull) break;
      --j;
    }
  }
  flags[blk] = (2ull << 62) | (excl + slot);
  p.blk_off[blk] = (int64_t)excl;
  p.blk_size[blk] = size;
  if (blk == p.n_blocks - 1) p.totals[0] = excl + slot;
  if (host) atomicAdd(p.totals + 1, 1ull);
  return (long long)excl;
}

// Payload checksum, every thread's share: the raw CRC of an odd-word-stride chunk, shifted to its position by one carry-less
// multiplication and XOR-reduced per warp into s_red[warp]. Call after the image is complete and a barrier.
template <int NT>
__device__ __forceinline__ void payload_crc_part(const Params &p, const uint32_t *img32, const uint32_t *tab, uint32_t size, uint32_t *s_red,
                                                 int tid, int lane, int warp) {
  const uint32_t len = size - kHeaderSize, W = len >> 2;
  uint32_t lw = (W + NT - 1u) / NT;
  lw |= 1u;   // odd word stride between the threads' chunks: bank-conflict free
  const int padw = (int)(NT * lw) - (int)W;   // leading zero words of the conceptual message
  const uint32_t *pay = img32 + kHeaderSize / 4u;
  uint32_t crc = 0;
  {
    const int w0 = tid * (int)lw - padw;
    for (int w = max(w0, 0); w < w0 + (int)lw; ++w) crc = crc_word(tab, crc, pay[w]);
  }
  if (crc != 0) crc = gf2_mulmod(crc, p.xpow32[(uint32_t)(NT - 1 - tid) * lw]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) crc ^= __shfl_xor_sync(0xffffffffu, crc, o);
  if (lane == 0) s_red[warp] = crc;
}

// Thread 0, after the barrier behind payload_crc_part: the payload crc's tail bytes, ObMicroBlockHeader
// (ob_micro_block_header.h:95-153) + its 16-bit checksum (ob_micro_block_header.cpp:193-233), then ONE bulk copy of the slot.
template <int NW>
__device__ __forceinline__ void finish_block(const Params &p, uint8_t *smem, const uint32_t *tab, const uint32_t *s_red, uint32_t size,
                                             uint32_t slot, uint32_t nrows, uint32_t ext_bit, uint32_t original, long long off) {
  uint32_t *img32 = reinterpret_cast<uint32_t *>(smem);
  const int nc = p.n_cols;
  const uint32_t len = size - kHeaderSize;
  uint32_t crc = 0;
  for (int w = 0; w < NW; ++w) crc ^= s_red[w];
  for (uint32_t k = len & ~3u; k < len; ++k) crc = crc_byte(tab, crc, smem[kHeaderSize + k]);
  const uint32_t ncu = (uint32_t)nc, rk = (uint32_t)p.rowkey_cnt, flag16 = 1u << 2;   // all_lob_in_row_
  const uint32_t opt = (ext_bit & 7u) << 3;                                            // row_index_byte 0, no var column
  const uint32_t row_data_off = size;                                                  // meta end == block end
  const uint16_t magic = (uint16_t)obf::MICRO_BLOCK_HEADER_MAGIC, version = (uint16_t)obf::MICRO_BLOCK_HEADER_VERSION;
  uint32_t cs = 0;
  auto f32 = [&](uint32_t x) { cs ^= (x & 0xffffu) ^ (x >> 16); };
  cs ^= magic;
  cs ^= version;
  cs ^= (uint32_t)obf::ENCODING_ROW_STORE;
  cs ^= opt;
  f32(ncu); f32(rk); f32(flag16 & 1u); f32(0u /*opt2_: var column count*/);
  f32(kHeaderSize); f32(nrows); f32(row_data_off); f32(original);
  f32(len); f32(len); f32(crc);   // 64-bit fields with a zero high half fold like 32-bit ones
  cs &= 0xffffu;
  img32[0] = (uint32_t)magic | ((uint32_t)version << 16);
  img32[1] = kHeaderSize;
  img32[2] = cs | (ncu << 16);
  img32[3] = rk | (flag16 << 16);
  img32[4] = nrows;
  img32[5] = (uint32_t)obf::ENCODING_ROW_STORE | (opt << 8);   // row_store_type_, opt_, opt2_ = 0
  img32[6] = row_data_off;
  img32[7] = original;
  img32[8] = 0u; img32[9] = 0u;                 // max_merged_trans_version_
  img32[10] = len;                              // data_length_
  img32[11] = len;                              // data_zlength_
  img32[12] = crc; img32[13] = 0u;              // data_checksum_
  img32[14] = 0u; img32[15] = 0u;               // column_checksums_ptr_
  // the other threads made their shared-memory writes visible to the async proxy before the barrier above
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  uint8_t *dst = p.image + off;
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(smem)), "r"(slot) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

template <bool CKSUM>
__global__ void __launch_bounds__(kThreads) obgpu_encode_blocks_kernel(const __grid_constant__ Params p) {
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t *img32 = reinterpret_cast<uint32_t *>(smem);                 // block image, p.slot_cap bytes
  uint32_t *tab = reinterpret_cast<uint32_t *>(smem + p.slot_cap);      // 4 x 256 crc tables
  // per column scratch behind the tables: [kWarps][n_cols] max, [kWarps][n_cols] NULL count, [n_cols] layout
  unsigned long long *s_wmax = reinterpret_cast<unsigned long long *>(smem + p.slot_cap + 4096u);
  uint32_t *s_wnull = reinterpret_cast<uint32_t *>(s_wmax + kWarps * p.n_cols);
  ColLayout *s_lay = reinterpret_cast<ColLayout *>(s_wnull + kWarps * p.n_cols);
  __shared__ uint32_t s_red[kWarps];
  __shared__ int s_blk;
  __shared__ uint32_t s_size, s_original, s_ext_bit, s_host;
  __shared__ long long s_off;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) s_blk = atomicAdd(p.ticket, 1);
  // zero image (cells are OR-ed in; padding up to the aligned slot must be zero): before anything else, under the ticket's round trip
  for (uint32_t i = (uint32_t)tid; i < p.slot_cap / 16u; i += kThreads) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  build_crc_tables<kThreads>(tab, tid);
  const int blk = s_blk;
  const int64_t row0 = (int64_t)blk * p.rows_per_block;
  const uint32_t nrows = (uint32_t)min(p.rows_per_block, p.total_rows - row0);
  const int nc = p.n_cols;
  __syncthreads();

  stats_pass<kThreads, CKSUM>(p, tab, row0, nrows, s_wmax, s_wnull, tid, lane, warp);
  __syncthreads();

  // ---- plan: warp 0, one lane per column (two rounds for more than 32 columns) -------------------------------------------
  if (warp == 0) {
    uint32_t at = kHeaderSize + 16u * (uint32_t)nc;
    unsigned long long original = 0;
    bool host = false;
    // ext bits: 1 as soon as any column has a NULL (ob_micro_block_encoder.cpp:507-517; a major merge leaves no NOP cell)
    bool any_null = false;
    for (int c = lane; c < nc; c += 32) {
      uint32_t n = 0;
      for (int w = 0; w < kWarps; ++w) n += s_wnull[w * nc + c];
      any_null = any_null || n != 0;
    }
    const uint32_t ext_bit = __any_sync(0xffffffffu, any_null) ? 1u : 0u;
    for (int cb = 0; cb < nc; cb += 32) {
      const int c = cb + lane;
      uint32_t bytes = 0, nn = 0;
      ColLayout l{};
      bool var = false;
      if (c < nc) {
        unsigned long long mx = 0;
        for (int w = 0; w < kWarps; ++w) { mx = max(mx, s_wmax[w * nc + c]); nn += s_wnull[w * nc + c]; }
        bool bp;
        const uint32_t size = packing_size(mx, p.col[c].byte_only == 0, bp);
        // ObRawEncoder::traverse (ob_raw_encoder.cpp:106-110,150-155): NULLs dominate -> var-stored column
        var = bp ? (unsigned long long)size * nn > (unsigned long long)nrows * 16ull : (unsigned long long)size * nn > (unsigned long long)nrows * 2ull;
        l.has_null = nn != 0;
        l.bp = bp;
        l.size = (uint8_t)size;
        l.attr = (uint8_t)(0x1u /*FIX_LENGTH*/ | (nn ? 0x2u /*HAS_EXTEND_VALUE*/ : 0u) | (bp ? 0x4u /*BIT_PACKING*/ : 0u));
        const unsigned long long bits = (nn ? (unsigned long long)ext_bit * nrows : 0ull) + (bp ? (unsigned long long)size * nrows : 0ull);
        l.bits_size = (uint32_t)((bits + 7ull) / 8ull);
        bytes = l.bits_size + (bp ? 0u : size * nrows);
      }
      uint32_t incl = bytes;   // column stores back to back: exclusive prefix over the columns
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
      }
      if (c < nc) {
        l.store_off = at + incl - bytes;
        s_lay[c] = l;
      }
      at += __shfl_sync(0xffffffffu, incl, 31);
      host = host || __any_sync(0xffffffffu, var);
      const uint32_t cells = c < nc ? (nrows - nn) * p.col[c].datum_len : 0u;
      original += __reduce_add_sync(0xffffffffu, cells);
    }
    if (lane == 0) {
      s_size = host ? 0u : at;
      s_original = (uint32_t)min(original, 0x7fffffffull);
      s_ext_bit = ext_bit;
      s_host = host;
      // publish the aligned size at once: the look-backs of the following blocks can pass over this one without waiting
      if (blk > 0) {
        volatile unsigned long long *flags = p.flags;
        flags[blk] = (1ull << 62) | (host ? 0ull : (unsigned long long)((at + p.align - 1u) & ~(p.align - 1u)));
      }
    }
  }
  __syncthreads();
  const uint32_t size = s_size;
  const uint32_t slot = (size + p.align - 1u) & ~(p.align - 1u);
  if (tid == 0) s_off = look_back(p, blk, size, slot, s_host != 0);

  if (size != 0) {
    // ---- pack ------------------------------------------------------------------------------------------------------------
    const uint32_t ext_bit = s_ext_bit;   // (the image was zeroed at the start of the kernel)
    if (tid < nc) {   // ObColumnHeader: version_, type_ (RAW = 0), attr_, obj_type_, extend_value_index_, offset_ (from the meta start), length_
      const ColLayout l = s_lay[tid];
      uint32_t *h = img32 + (kHeaderSize + 16u * (uint32_t)tid) / 4u;
      h[0] = ((uint32_t)l.attr << 16) | ((uint32_t)p.col[tid].obj_type << 24);
      h[1] = 0u;
      h[2] = l.store_off - (kHeaderSize + 16u * (uint32_t)nc);
      h[3] = l.size;
    }
    for (int c = 0; c < nc; ++c) {
      const ColSpec &cs = p.col[c];
      const ColLayout l = s_lay[c];
      const int64_t *v = cs.vals + row0;
      const uint8_t *nl = (cs.nulls && l.has_null) ? cs.nulls + row0 : nullptr;
      const uint32_t bit0 = l.store_off * 8u;                                    // block bit address of the bit area
      const uint32_t val0 = bit0 + (l.has_null ? ext_bit * nrows : 0u);         // bit-packed values follow the ext bits
      for (uint32_t r = (uint32_t)tid; r < nrows; r += kThreads) {
        if (nl && nl[r] != 0) {
          const uint32_t b = bit0 + r * ext_bit;   // STORED_NULL = 1
          atomicOr(img32 + (b >> 5), 1u << (b & 31u));
          continue;
        }
        const unsigned long long x = (unsigned long long)v[r] & cs.store_mask;
        // bit-packed cells: size bits each behind the ext bits; byte-packed cells: 8 * size bits each behind the bit area
        const uint32_t w = l.bp ? l.size : 8u * l.size;
        or_bits(img32, (l.bp ? val0 : (l.store_off + l.bits_size) * 8u) + r * w, w, x);
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // pack writes -> visible to the bulk copy issued by thread 0
    __syncthreads();
    payload_crc_part<kThreads>(p, img32, tab, size, s_red, tid, lane, warp);
  }
  __syncthreads();

  if (tid == 0 && size != 0) finish_block<kWarps>(p, smem, tab, s_red, size, slot, nrows, s_ext_bit, s_original, s_off);
}

// Column checksums alone (ObMicroBlockChecksumHelper::cal_column_checksum over plain columns).
constexpr int kCkThreads = 256;
__global__ void __launch_bounds__(kCkThreads) obgpu_column_checksum_kernel(const __grid_constant__ Params p) {
  __shared__ uint32_t tab[1024];
  const int tid = threadIdx.x, lane = tid & 31;
  {
    uint32_t c = (uint32_t)tid;
#pragma unroll
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? kCrcPoly ^ (c >> 1) : c >> 1;
    tab[tid] = c;
  }
  __syncthreads();
  {
    uint32_t c = tab[tid];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      c = (c >> 8) ^ tab[c & 0xffu];
      tab[k * 256 + tid] = c;
    }
  }
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * kCkThreads;
  for (int c = 0; c < p.n_cols; ++c) {
    const ColSpec &cs = p.col[c];
    const uint32_t len_crc = crc_word(tab, 0u, (uint32_t)cs.datum_len), null_crc = crc_word(tab, 0u, 0x80000000u);
    unsigned long long sum = 0;
    for (int64_t r = (int64_t)blockIdx.x * kCkThreads + tid; r < p.total_rows; r += stride) {
      uint32_t crc = null_crc;
      if (!(cs.nulls && cs.nulls[r] != 0)) {
        const unsigned long long x = (unsigned long long)cs.vals[r];
        crc = len_crc;
        if (cs.datum_len == 8) {
          crc = crc_word(tab, crc, (uint32_t)x);
          crc = crc_word(tab, crc, (uint32_t)(x >> 32));
        } else if (cs.datum_len == 4) {
          crc = crc_word(tab, crc, (uint32_t)x);
        } else {
          for (uint32_t k = 0; k < cs.datum_len; ++k) crc = crc_byte(tab, crc, (uint32_t)(x >> (8u * k)) & 0xffu);
        }
      }
      sum += crc;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0 && sum != 0) atomicAdd(p.checksums + c, sum);
  }
}

}  // namespace enc

struct obgpu_encoded {
  obgpu_ctx *ctx = nullptr;
  void *arena = nullptr;
  uint8_t *d_image = nullptr;
  int64_t *d_off = nullptr;
  uint32_t *d_size = nullptr;
  unsigned long long *d_checksums = nullptr, *d_totals = nullptr;
  int32_t n_cols = 0, n_blocks = 0;
  int64_t total_rows = 0;
  bool info_valid = false;
  obgpu_encoded_info info{};
};

// x^(32 k) mod P for every k a chunk shift can take (a CTA's shared memory bounds the block image), built once per device
static const uint32_t *enc_xpow_table(obgpu_ctx *ctx) {
  static std::mutex mu;
  static std::map<int, uint32_t *> tables;
  std::lock_guard<std::mutex> g(mu);
  auto it = tables.find(ctx->device);
  if (it != tables.end()) return it->second;
  // the RAW kernel's 128 threads and the codec kernel's 256 (encode_codecs.cuh) index it as (threads - 1 - tid) * chunk words
  size_t n_pow = 1;
  for (const size_t nt : {(size_t)enc::kThreads, (size_t)2 * enc::kThreads}) {
    const size_t lw_cap = (size_t)((ctx->max_smem_optin / 4 + nt - 1) / nt) | 1;
    n_pow = std::max(n_pow, (nt - 1) * lw_cap + 1);
  }
  std::vector<uint32_t> xpow(n_pow);
  uint32_t b = 0x80000000u;
  for (size_t k = 0; k < n_pow; ++k) {
    xpow[k] = b;
    for (int i = 0; i < 32; ++i) b = (b >> 1) ^ ((b & 1u) ? enc::kCrcPoly : 0u);
  }
  uint32_t *d = nullptr;
  if (cudaMalloc((void **)&d, n_pow * 4) != cudaSuccess) return nullptr;
  if (cudaMemcpy(d, xpow.data(), n_pow * 4, cudaMemcpyHostToDevice) != cudaSuccess) { cudaFree(d); return nullptr; }
  tables[ctx->device] = d;
  return d;
}

static int enc_fill_cols(enc::Params &p, const obgpu_encode_col *cols, int32_t n_cols) {
  for (int c = 0; c < n_cols; ++c) {
    const int sc = obf::store_class_of((uint8_t)cols[c].obj_type);
    if ((sc != 1 && sc != 2) || !cols[c].dev_vals) return sc == 5 ? OBGPU_NOT_SUPPORTED : OBGPU_INVALID_ARGUMENT;
    enc::ColSpec &s = p.col[c];
    s.vals = cols[c].dev_vals;
    s.nulls = cols[c].dev_null;
    s.store_mask = obf::low_mask((uint32_t)obf::type_store_size((uint8_t)cols[c].obj_type) * 8u);
    s.obj_type = (uint8_t)cols[c].obj_type;
    s.byte_only = cols[c].byte_packing_only ? 1 : 0;
    s.datum_len = (uint8_t)obf::datum_len_of((uint8_t)cols[c].obj_type);
    s.sc = (uint8_t)sc;
    s.ts = (uint8_t)obf::type_store_size((uint8_t)cols[c].obj_type);
  }
  p.n_cols = n_cols;
  return OBGPU_SUCCESS;
}

// Checks the call's shape, fills p.col and allocates the handle's arena (flags, offsets, sizes, image of n_blocks slots) on the
// context's stream; the caller sets the encodings and launches.
static int enc_prepare(obgpu_ctx *ctx, const obgpu_encode_col *cols, int32_t n_cols, int32_t rowkey_col_cnt, int64_t total_rows,
                       int64_t rows_per_block, int32_t align, enc::Params &p, int64_t &n_blocks64) {
  if (!ctx || !cols || n_cols <= 0 || n_cols > enc::kMaxCols || rowkey_col_cnt < 0 || rowkey_col_cnt > n_cols || total_rows <= 0 ||
      rows_per_block <= 0 || rows_per_block > (1 << 22) || align < 16 || align > 4096 || (align & (align - 1)) != 0)
    return OBGPU_INVALID_ARGUMENT;
  n_blocks64 = (total_rows + rows_per_block - 1) / rows_per_block;
  if (n_blocks64 > 0x7fffffff) return OBGPU_NOT_SUPPORTED;
  return enc_fill_cols(p, cols, n_cols);
}

static int enc_alloc(obgpu_ctx *ctx, enc::Params &p, int32_t n_cols, int32_t rowkey_col_cnt, int64_t total_rows, int64_t rows_per_block,
                     int32_t align, int64_t n_blocks64, int64_t slot_cap, obgpu_encoded **out) {
  const uint32_t lw_max = (uint32_t)(((slot_cap / 4 + enc::kThreads - 1) / enc::kThreads) | 1);
  const uint32_t *d_xpow = enc_xpow_table(ctx);
  if (!d_xpow) return OBGPU_ALLOCATE_MEMORY_FAILED;
  obgpu_encoded *e = new obgpu_encoded();
  e->ctx = ctx;
  e->n_cols = n_cols;
  e->n_blocks = (int32_t)n_blocks64;
  e->total_rows = total_rows;
  auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o = 0;
  const size_t o_ctl = o; o += al(256 + (size_t)n_cols * 8);
  const size_t o_flags = o; o += al((size_t)n_blocks64 * 8);
  const size_t o_off = o; o += al((size_t)n_blocks64 * 8);
  const size_t o_size = o; o += al((size_t)n_blocks64 * 4);
  const size_t o_img = o; o += al((size_t)n_blocks64 * (size_t)slot_cap);
  cudaError_t err = cudaMallocAsync(&e->arena, o, ctx->stream);
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); delete e; return OBGPU_ALLOCATE_MEMORY_FAILED; }
  uint8_t *a = (uint8_t *)e->arena;
  e->d_totals = (unsigned long long *)(a + o_ctl);
  e->d_checksums = (unsigned long long *)(a + o_ctl + 256);
  e->d_off = (int64_t *)(a + o_off);
  e->d_size = (uint32_t *)(a + o_size);
  e->d_image = a + o_img;
  cudaMemsetAsync(a, 0, o_off, ctx->stream);   // totals, ticket, checksums, look-back flags
  p.rowkey_cnt = rowkey_col_cnt;
  p.n_blocks = e->n_blocks;
  p.want_checksums = 1;
  p.total_rows = total_rows;
  p.rows_per_block = rows_per_block;
  p.align = (uint32_t)align;
  p.slot_cap = (uint32_t)slot_cap;
  p.lw_max = lw_max;
  p.image = e->d_image;
  p.blk_off = e->d_off;
  p.blk_size = e->d_size;
  p.flags = (unsigned long long *)(a + o_flags);
  p.checksums = e->d_checksums;
  p.totals = e->d_totals;
  p.ticket = (int32_t *)(a + o_ctl + 128);
  p.xpow32 = d_xpow;
  *out = e;
  return OBGPU_SUCCESS;
}

// every column RAW: obgpu_encode_blocks_kernel
static int enc_launch_raw(obgpu_ctx *ctx, enc::Params &p, int32_t n_cols, int32_t rowkey_col_cnt, int64_t total_rows, int64_t rows_per_block,
                          int32_t align, int64_t n_blocks64, obgpu_encoded **out) {
  // the largest block: every column 8 bytes wide + one ext bit per cell
  const int64_t bound = (int64_t)enc::kHeaderSize + 16 * n_cols + (int64_t)n_cols * (rows_per_block * 8 + (rows_per_block + 7) / 8 + 1);
  const int64_t slot_cap = (bound + align - 1) / align * align;
  const size_t smem = (size_t)slot_cap + 4096 + (size_t)n_cols * (enc::kWarps * 12 + sizeof(enc::ColLayout)) + 16;
  if ((int64_t)smem > (int64_t)ctx->max_smem_optin - 8192) return OBGPU_NOT_SUPPORTED;   // block image does not fit one CTA's shared memory
  cudaSetDevice(ctx->device);
  obgpu_encoded *e = nullptr;
  int rc = enc_alloc(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, &e);
  if (rc != OBGPU_SUCCESS) return rc;
  cudaError_t err = cudaFuncSetAttribute(enc::obgpu_encode_blocks_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); obgpu_encoded_free(e); return OBGPU_ERR_SYS; }
  enc::obgpu_encode_blocks_kernel<true><<<(unsigned)e->n_blocks, enc::kThreads, smem, ctx->stream>>>(p);
  ctx->launches++;
  err = cudaGetLastError();
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); obgpu_encoded_free(e); return OBGPU_ERR_SYS; }
  *out = e;
  return OBGPU_SUCCESS;
}

extern "C" {

int obgpu_encode_columns(obgpu_ctx *ctx, const obgpu_encode_col *cols, int32_t n_cols, int32_t rowkey_col_cnt, int64_t total_rows,
                         int64_t rows_per_block, int32_t align, obgpu_encoded **out) {
  return obgpu_encode_columns_with(ctx, cols, nullptr, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, out);
}

int obgpu_encoded_get_info(obgpu_encoded *e, obgpu_encoded_info *info) {
  if (!e || !info) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = e->ctx;
  if (!e->info_valid) {
    cudaSetDevice(ctx->device);
    unsigned long long *hp = (unsigned long long *)ctx->h_pinned;
    CUDA_TRY(ctx, cudaMemcpyAsync(hp, e->d_totals, 16, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    e->info.image_size = (int64_t)hp[0];
    e->info.n_host_blocks = (int32_t)hp[1];
    e->info.n_blocks = e->n_blocks;
    e->info.total_rows = e->total_rows;
    e->info_valid = true;
  }
  *info = e->info;
  return OBGPU_SUCCESS;
}

int obgpu_encoded_fetch(obgpu_encoded *e, void *host_image, int64_t image_cap, int64_t *host_offsets, int64_t *host_sizes, int32_t blocks_cap) {
  if (!e) return OBGPU_INVALID_ARGUMENT;
  obgpu_encoded_info info;
  int rc = obgpu_encoded_get_info(e, &info);
  if (rc != OBGPU_SUCCESS) return rc;
  obgpu_ctx *ctx = e->ctx;
  if ((host_image && image_cap < info.image_size) || ((host_offsets || host_sizes) && blocks_cap < info.n_blocks)) return OBGPU_BUF_NOT_ENOUGH;
  if (host_image && info.image_size > 0) CUDA_TRY(ctx, cudaMemcpyAsync(host_image, e->d_image, (size_t)info.image_size, cudaMemcpyDeviceToHost, ctx->stream));
  if (host_offsets) CUDA_TRY(ctx, cudaMemcpyAsync(host_offsets, e->d_off, (size_t)info.n_blocks * 8, cudaMemcpyDeviceToHost, ctx->stream));
  std::vector<uint32_t> sz;
  if (host_sizes) {
    sz.resize((size_t)info.n_blocks);
    CUDA_TRY(ctx, cudaMemcpyAsync(sz.data(), e->d_size, (size_t)info.n_blocks * 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (host_sizes) for (int32_t i = 0; i < info.n_blocks; ++i) host_sizes[i] = sz[(size_t)i];
  return OBGPU_SUCCESS;
}

int obgpu_encoded_device_image(obgpu_encoded *e, const void **dev_image, const int64_t **dev_offsets, const uint32_t **dev_sizes) {
  if (!e) return OBGPU_INVALID_ARGUMENT;
  if (dev_image) *dev_image = e->d_image;
  if (dev_offsets) *dev_offsets = e->d_off;
  if (dev_sizes) *dev_sizes = e->d_size;
  return OBGPU_SUCCESS;
}

int obgpu_encoded_column_checksums(obgpu_encoded *e, int64_t *host_checksums) {
  if (!e || !host_checksums) return OBGPU_INVALID_ARGUMENT;
  obgpu_ctx *ctx = e->ctx;
  cudaSetDevice(ctx->device);
  CUDA_TRY(ctx, cudaMemcpyAsync(host_checksums, e->d_checksums, (size_t)e->n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  return OBGPU_SUCCESS;
}

void obgpu_encoded_free(obgpu_encoded *e) {
  if (!e) return;
  if (e->arena) {
    cudaSetDevice(e->ctx->device);
    cudaFreeAsync(e->arena, e->ctx->stream);
  }
  delete e;
}

int obgpu_column_checksums(obgpu_ctx *ctx, const obgpu_encode_col *cols, int32_t n_cols, int64_t total_rows, int64_t *host_checksums) {
  if (!ctx || !cols || !host_checksums || n_cols <= 0 || n_cols > enc::kMaxCols || total_rows < 0) return OBGPU_INVALID_ARGUMENT;
  enc::Params p{};
  int rc = enc_fill_cols(p, cols, n_cols);
  if (rc != OBGPU_SUCCESS) return rc;
  cudaSetDevice(ctx->device);
  unsigned long long *d = nullptr;
  CUDA_TRY(ctx, cudaMallocAsync((void **)&d, (size_t)n_cols * 8, ctx->stream));
  cudaMemsetAsync(d, 0, (size_t)n_cols * 8, ctx->stream);
  p.total_rows = total_rows;
  p.checksums = d;
  const int64_t want = (total_rows + enc::kCkThreads * 8 - 1) / (enc::kCkThreads * 8);
  const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)ctx->sm_count * 8));
  enc::obgpu_column_checksum_kernel<<<grid, enc::kCkThreads, 0, ctx->stream>>>(p);
  ctx->launches++;
  cudaError_t err = cudaMemcpyAsync(host_checksums, d, (size_t)n_cols * 8, cudaMemcpyDeviceToHost, ctx->stream);
  if (err == cudaSuccess) err = cudaStreamSynchronize(ctx->stream);
  cudaFreeAsync(d, ctx->stream);
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); return OBGPU_ERR_SYS; }
  return OBGPU_SUCCESS;
}

int obgpu_merge_result_encode(obgpu_merge_result *res, const int32_t *result_cols, const int32_t *obj_types, int32_t n_cols,
                              int32_t rowkey_col_cnt, int64_t rows_per_block, int32_t align, obgpu_encoded **out) {
  return obgpu_merge_result_encode_with(res, result_cols, obj_types, nullptr, n_cols, rowkey_col_cnt, rows_per_block, align, out);
}

int obgpu_merge_result_encode_with(obgpu_merge_result *res, const int32_t *result_cols, const int32_t *obj_types, const int32_t *encodings,
                                   int32_t n_cols, int32_t rowkey_col_cnt, int64_t rows_per_block, int32_t align, obgpu_encoded **out) {
  if (!res || !result_cols || !obj_types || n_cols <= 0 || n_cols > enc::kMaxCols || !out) return OBGPU_INVALID_ARGUMENT;
  obgpu_merge_info info;
  int rc = obgpu_merge_result_info(res, &info);
  if (rc != OBGPU_SUCCESS) return rc;
  if (info.out_rows <= 0) return OBGPU_INVALID_ARGUMENT;
  std::vector<obgpu_encode_col> cols((size_t)n_cols);
  for (int i = 0; i < n_cols; ++i) {
    obgpu_encode_col &c = cols[(size_t)i];
    c.obj_type = obj_types[i];
    c.byte_packing_only = 0;
    const int32_t k = result_cols[i];
    if (k == -1) { c.dev_vals = res->d_out_key; c.dev_null = nullptr; }
    else if (k < -1) {
      const size_t m = (size_t)(-k - 2);
      if (m >= res->out_more.size()) return OBGPU_INVALID_ARGUMENT;
      c.dev_vals = res->out_more[m];
      c.dev_null = nullptr;
    } else {
      if (k >= res->n_cols) return OBGPU_INVALID_ARGUMENT;
      if (!res->col_is_string.empty() && res->col_is_string[(size_t)k]) return OBGPU_NOT_SUPPORTED;
      c.dev_vals = res->out_vals[(size_t)k];
      c.dev_null = res->out_null[(size_t)k];
    }
  }
  return obgpu_encode_columns_with(res->ctx, cols.data(), encodings, n_cols, rowkey_col_cnt, info.out_rows, rows_per_block, align, out);
}

}  // extern "C"
