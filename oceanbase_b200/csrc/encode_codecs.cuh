// Phase B with codecs: PAX micro-blocks whose integer columns are DICT / RLE / CONST / INTEGER_BASE_DIFF / RAW -- forced per
// column, or chosen per micro-block (OBGPU_ENC_AUTO) -- byte for byte the blocks the host writer builds for the same rows and
// encodings (sstable_writer.cpp: BlockBuilder::encode_raw / encode_dict / encode_rle / encode_const / encode_base_diff and
// choose_auto_encoding, which are the specification restated here). Same outer shape as the RAW kernel (encode_kernels.cuh):
// one CTA per micro-block, ticket + decoupled look-back, the stats pass with the column checksums, parallel crc32c, one bulk
// store. Per column, in column order, over scratch reused from column to column (so shared memory grows with the rows of a
// block, not with rows x columns):
//
//   keys    : the non-NULL store images, as build_int_dict(sorted) orders them (x ^ sign for the signed class), minus the block
//             minimum, compacted in row order together with their row (u16)
//   sort    : cub::BlockRadixSort over bit_width(max - min) bits (stable: the first element of an equal run is the value's first
//             occurrence); a single value or no value skips it
//   derive  : adjacent compare + block scans: sorted dictionary (head positions), sorted ref per row (NULL -> count), per value
//             counts and the most frequent one, first-occurrence order (RLE's dictionary), run count and last run start
//   choose  : OBGPU_ENC_AUTO runs choose_auto_encoding's formulas literally
//   pack    : the codec's meta and cells at the column's offset; every byte goes in through the shared atomicOr of or_bits, so
//             meta and cells that share a word need no ordering between them
//
// A block whose codec the host writer refuses (a forced codec on data it does not take, or RAW with NULL-dominated cells) reads
// size 0 and is left to the host writer, like the RAW kernel's var-stored blocks.
#pragma once
#include <cub/block/block_radix_sort.cuh>

namespace enc {

constexpr int kCodecThreads = 256;
constexpr int kCodecWarps = kCodecThreads / 32;
// Rows per block the codec kernel takes. With at most 4096 rows, RLE's runs x row_id_byte stays <= 8192 (<= 32767, the int16
// ObRLEDecoder keeps it in), and a CONST column with <= 32 exceptions has <= 33 dictionary values and a meta far below 64 KiB:
// the host writer's refusals for those limits cannot occur here.
constexpr int kCodecMaxRows = 4096;

__host__ __device__ __forceinline__ uint32_t byte_packed_size(unsigned long long v) {   // get_byte_packed_int_size
  return v <= 0xffull ? 1u : v <= 0xffffull ? 2u : v <= 0xffffffffull ? 4u : 8u;
}
__device__ __forceinline__ uint32_t bit_width_of(unsigned long long v) { return v == 0 ? 1u : 64u - (uint32_t)__clzll((long long)v); }
__device__ __forceinline__ uint32_t int_size_bytes(unsigned long long v) { return (bit_width_of(v) + 7u) / 8u; }   // get_int_size

template <int ITEMS>
using CodecSort = cub::BlockRadixSort<unsigned long long, kCodecThreads, ITEMS, uint16_t>;

// Shared memory of the codec kernel behind the block image (slot_cap) and the crc tables (4096): the sort's storage (aliased by
// the sorted keys), [warps][n_cols] max + NULL count, and per row / per value u16 arrays + a flag byte.
template <int ITEMS>
__host__ __device__ constexpr size_t codec_sort_bytes() {
  return ((sizeof(typename CodecSort<ITEMS>::TempStorage) > 8u * kCodecThreads * ITEMS ? sizeof(typename CodecSort<ITEMS>::TempStorage)
                                                                                       : 8u * kCodecThreads * ITEMS) + 15u) & ~(size_t)15u;
}
template <int ITEMS>
__host__ __device__ constexpr size_t codec_scratch_bytes(int n_cols) {
  return codec_sort_bytes<ITEMS>() + (size_t)n_cols * kCodecWarps * 12u + 2u * (4u * kCodecThreads * ITEMS + 8u) + kCodecThreads * ITEMS;
}

template <int NT>
__device__ __forceinline__ uint32_t block_excl_sum(uint32_t x, uint32_t *s_w, uint32_t &total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t incl = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += u;
  }
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  uint32_t before = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < NT / 32; ++w) {
    const uint32_t v = s_w[w];
    before += w < warp ? v : 0u;
    tot += v;
  }
  __syncthreads();
  total = tot;
  return before + incl - x;
}

template <int NT, int K>
__device__ __forceinline__ void block_max(unsigned long long (&v)[K], unsigned long long *s_w /* [K][NT / 32] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] = max(v[k], __shfl_xor_sync(0xffffffffu, v[k], o));
    if (lane == 0) s_w[k * (NT / 32) + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    unsigned long long m = 0;
#pragma unroll
    for (int w = 0; w < NT / 32; ++w) m = max(m, s_w[k * (NT / 32) + w]);
    v[k] = m;
  }
  __syncthreads();
}

// What choose_auto_encoding reads of a column (no NOP cells: the device encodes merged rows).
struct ColFacts {
  int64_t n, null_cnt, distinct, max_cnt, runs, last_run, exc_max_row;
  unsigned long long max_integer, tmin, tmax;   // tmin / tmax: key order (x ^ sign for the signed class)
  int ts, sc, ext_bit;
  bool enable_bp;
};

__device__ __forceinline__ int64_t packing_size64(unsigned long long v, bool enable_bp, bool &bp) { return (int64_t)packing_size(v, enable_bp, bp); }

// choose_auto_encoding (sstable_writer.cpp), integer columns without NOP cells: the same integer formulas, candidate order,
// strict replacements, raw_size / 4 stop and distinct <= n / 2 gate. The CONST candidate takes the most frequent value with the
// lowest sorted index where the host takes the lowest first-seen index; the two differ only on a tie, and a tie with at most
// max(n / 10, 1) exceptions needs n <= 2, where both exception rows fit one row-id byte: the sizes are the same.
__device__ int choose_auto(const ColFacts &f) {
  const int64_t n = f.n, ts = f.ts, null_cnt = f.null_cnt, ext_cnt = f.null_cnt, distinct = f.distinct;
  const int64_t ext_store = (ext_cnt > 0) ? (n * f.ext_bit + 1) / 8 : 0;
  int64_t raw_size;
  {
    int64_t bp_len = 0, fix_len = 0, raw_var = 0;
    bool is_var = false, bp = false;
    const int64_t size = packing_size64(f.max_integer, f.enable_bp, bp);
    if (bp) {
      if (size * ext_cnt > n * 2 * 8) { is_var = true; raw_var = (size / 8 + 1) * (n - ext_cnt); }
      else bp_len = size;
    } else {
      fix_len = size;
    }
    if (fix_len > 0 && bp_len == 0 && fix_len * ext_cnt > n * 2) { is_var = true; fix_len = 0; }
    raw_size = bp_len > 0 ? bp_len * n / 8 + 1 : (!is_var ? fix_len * n : raw_var + n * 2);
    raw_size += ext_store;
  }
  const int64_t dict_fix = f.enable_bp ? int_size_bytes(f.max_integer) : byte_packed_size(f.max_integer);
  const int64_t dict_meta = 9 + dict_fix * distinct;
  int64_t max_ref = distinct - 1;
  if (null_cnt > 0) max_ref = distinct;
  int64_t dict_size;
  {
    bool bp = false;
    const int64_t size = packing_size64((unsigned long long)max(max_ref, (int64_t)0), f.enable_bp, bp);
    dict_size = dict_meta + (bp ? (n * size + 7) / 8 : n * size);
  }
  bool const_ok = true;
  int64_t const_size = 0;
  {
    const int64_t max_cnt = max(f.max_cnt, null_cnt);
    const int64_t exc = n - max_cnt;
    if (exc > 32 || exc > max(n * 10 / 100, (int64_t)1)) {
      const_ok = false;
    } else if (exc == 0) {
      const_size = (null_cnt == 0 ? ts : 0) + 6;
    } else {
      const_size = 6 + dict_meta + exc * (byte_packed_size((unsigned long long)f.exc_max_row) + 1);
    }
  }
  if (distinct <= 1 && const_ok) return OBGPU_ENC_CONST;
  int choose = OBGPU_ENC_RAW;
  int64_t choose_size = raw_size;
  const int64_t acceptable = raw_size / 4;
  if (dict_size < choose_size) { choose = OBGPU_ENC_DICT; choose_size = dict_size; }
  if (distinct <= n / 2) {
    const int64_t rle_size = 10 + dict_meta + f.runs * (byte_packed_size((unsigned long long)f.last_run) + byte_packed_size((unsigned long long)max(max_ref, (int64_t)0)));
    if (rle_size < choose_size) { choose = OBGPU_ENC_RLE; choose_size = rle_size; }
    if (const_ok && const_size < choose_size) { choose = OBGPU_ENC_CONST; choose_size = const_size; }
  }
  if (choose_size <= acceptable) return choose;
  if (null_cnt < n) {
    // min / max of the sign-extended images: key order minus the sign bit; a negative minimum makes the original width 64 bits
    const unsigned long long sign = f.sc == 1 ? 1ull << (8 * f.ts - 1) : 0ull;
    const unsigned long long delta = f.tmax - f.tmin;
    const unsigned long long max_unsigned = f.sc == 1 ? ((f.tmin < sign) ? ~0ull : (f.tmax ^ sign)) : f.tmax;
    if (delta != 0) {
      bool bp = false;
      int64_t orig = packing_size64(max_unsigned, true, bp);
      if (!bp) orig *= 8;
      bp = false;
      int64_t dsz = packing_size64(delta, true, bp);
      if (!bp) dsz *= 8;
      if ((orig - dsz) * n > (2 + ts) * 8) {
        const int64_t bd_size = (bp ? (n * dsz + 7) / 8 : n * (dsz / 8)) + 2 + ts;
        if (bd_size < choose_size) { choose = OBGPU_ENC_INTEGER_BASE_DIFF; choose_size = bd_size; }
      }
    }
  }
  return choose;
}

template <int ITEMS>
__global__ void __launch_bounds__(kCodecThreads) obgpu_encode_codecs_kernel(const __grid_constant__ Params p) {
  constexpr int NT = kCodecThreads, NW = kCodecWarps, CAP = NT * ITEMS;
  using Sort = CodecSort<ITEMS>;
  extern __shared__ __align__(128) uint8_t smem[];
  uint32_t *img32 = reinterpret_cast<uint32_t *>(smem);
  uint32_t *tab = reinterpret_cast<uint32_t *>(smem + p.slot_cap);
  uint8_t *scr = smem + p.slot_cap + 4096u;
  typename Sort::TempStorage &s_sort = *reinterpret_cast<typename Sort::TempStorage *>(scr);
  unsigned long long *s_key = reinterpret_cast<unsigned long long *>(scr);   // aliases the sort's storage: staged keys, then sorted keys
  scr += codec_sort_bytes<ITEMS>();
  const int nc = p.n_cols;
  unsigned long long *s_wmax = reinterpret_cast<unsigned long long *>(scr);
  uint32_t *s_wnull = reinterpret_cast<uint32_t *>(s_wmax + NW * nc);
  uint16_t *s_row = reinterpret_cast<uint16_t *>(s_wnull + NW * nc);   // staged / sorted position -> row
  uint16_t *s_ref = s_row + CAP;                                        // row -> sorted ref (NULL: count)
  uint16_t *s_hpos = s_ref + CAP;                                       // sorted ref -> first sorted position, [count] = non-NULL rows
  uint16_t *s_fo = s_hpos + CAP + 4;                                    // sorted ref -> first-occurrence ref
  uint8_t *s_flag = reinterpret_cast<uint8_t *>(s_fo + CAP + 4);        // row: 1 NULL, 2 first occurrence of its value
  __shared__ uint32_t s_w32[NW], s_red[NW];
  __shared__ unsigned long long s_w64[2 * NW];
  __shared__ int s_blk;
  __shared__ long long s_off;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) s_blk = atomicAdd(p.ticket, 1);
  for (uint32_t i = (uint32_t)tid; i < p.slot_cap / 16u; i += NT) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0u, 0u, 0u, 0u);
  build_crc_tables<NT>(tab, tid);
  const int blk = s_blk;
  const int64_t row0 = (int64_t)blk * p.rows_per_block;
  const uint32_t n = (uint32_t)min(p.rows_per_block, p.total_rows - row0);
  __syncthreads();
  stats_pass<NT, true>(p, tab, row0, n, s_wmax, s_wnull, tid, lane, warp);
  __syncthreads();

  uint32_t ext_bit = 0;   // 1 as soon as any column has a NULL (ob_micro_block_encoder.cpp:507-517)
  for (int i = 0; i < NW * nc; ++i) ext_bit |= s_wnull[i] != 0 ? 1u : 0u;
  const uint32_t meta0 = kHeaderSize + 16u * (uint32_t)nc;
  uint32_t at = meta0;
  unsigned long long original = 0;
  bool host = false;

  for (int c = 0; c < nc && !host; ++c) {
    const ColSpec &cs = p.col[c];
    unsigned long long max_integer = 0;
    uint32_t null_cnt = 0;
    for (int w = 0; w < NW; ++w) { max_integer = max(max_integer, s_wmax[w * nc + c]); null_cnt += s_wnull[w * nc + c]; }
    original += (unsigned long long)(n - null_cnt) * cs.datum_len;
    const uint32_t nn = n - null_cnt, ts = cs.ts;
    const bool enable_bp = cs.byte_only == 0, has_null = null_cnt != 0;
    const unsigned long long sign = cs.sc == 1 ? 1ull << (8u * ts - 1u) : 0ull;
    const int64_t *vals = cs.vals + row0;
    const uint8_t *nulls = cs.nulls ? cs.nulls + row0 : nullptr;
    const int want = cs.enc;
    const bool need_dict = want != OBGPU_ENC_RAW && want != OBGPU_ENC_INTEGER_BASE_DIFF;

    // ---- keys: min / max in key order, compacted non-NULL rows ---------------------------------------------------------------
    unsigned long long tmin = 0, tmax = 0;
    uint32_t cnt = 0, runs = 1, last_run = 0, exc_max_row = 0, max_cnt = 0, const_ref = 0, run_before = 0, exc_before = 0;
    if (want != OBGPU_ENC_RAW) {
      unsigned long long key[ITEMS];
      uint32_t okm = 0, nok = 0;
      unsigned long long mm[2] = {0ull, 0ull};   // max key, max ~key
#pragma unroll
      for (int i = 0; i < ITEMS; ++i) {
        const uint32_t r = (uint32_t)tid * ITEMS + i;
        key[i] = 0;
        if (r < n) {
          const bool is_null = nulls && nulls[r] != 0;
          s_flag[r] = is_null ? 1 : 0;
          if (!is_null) {
            key[i] = ((unsigned long long)vals[r] & cs.store_mask) ^ sign;
            okm |= 1u << i;
            ++nok;
            mm[0] = max(mm[0], key[i]);
            mm[1] = max(mm[1], ~key[i]);
          }
        }
      }
      block_max<NT, 2>(mm, s_w64);
      if (nn != 0) { tmax = mm[0]; tmin = ~mm[1]; }
      if (need_dict) {
        uint32_t tot;
        uint32_t q = block_excl_sum<NT>(nok, s_w32, tot);
#pragma unroll
        for (int i = 0; i < ITEMS; ++i)
          if ((okm >> i) & 1u) { s_key[q] = key[i] - tmin; s_row[q] = (uint16_t)(tid * ITEMS + i); ++q; }
        __syncthreads();
        uint16_t rowv[ITEMS];
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t q2 = (uint32_t)tid * ITEMS + i;
          key[i] = q2 < nn ? s_key[q2] : ~0ull;   // padding sorts behind every key: stable, and placed after them
          rowv[i] = q2 < nn ? s_row[q2] : (uint16_t)0;
        }
        __syncthreads();
        const unsigned long long range = tmax - tmin;
        if (range != 0) {
          Sort(s_sort).Sort(key, rowv, 0, (int)bit_width_of(range));
          __syncthreads();
#pragma unroll
          for (int i = 0; i < ITEMS; ++i) { s_key[tid * ITEMS + i] = key[i]; s_row[tid * ITEMS + i] = rowv[i]; }
          __syncthreads();
        }
        // ---- heads of equal runs: sorted dictionary, sorted refs ---------------------------------------------------------
        uint32_t heads = 0, hm = 0;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t q2 = (uint32_t)tid * ITEMS + i;
          const bool h = q2 < nn && (q2 == 0 || s_key[q2] != s_key[q2 - 1]);
          hm |= (h ? 1u : 0u) << i;
          heads += h ? 1u : 0u;
        }
        uint32_t d = block_excl_sum<NT>(heads, s_w32, cnt);
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t q2 = (uint32_t)tid * ITEMS + i;
          if (q2 < nn) {
            const uint32_t r = s_row[q2];
            if ((hm >> i) & 1u) { s_hpos[d] = (uint16_t)q2; s_flag[r] |= 2; ++d; }
            s_ref[r] = (uint16_t)(d - 1);
          }
          const uint32_t r = (uint32_t)tid * ITEMS + i;
          if (r < n && (s_flag[r] & 1)) s_ref[r] = (uint16_t)cnt;
        }
        if (tid == 0) s_hpos[cnt] = (uint16_t)nn;
        __syncthreads();
        // ---- first occurrences, runs, most frequent value ----------------------------------------------------------------
        uint32_t firsts = 0, bnd = 0;
        unsigned long long m2[2] = {0ull, 0ull};   // (count << 32 | ~sorted ref): max count, lowest ref; last run start
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t r = (uint32_t)tid * ITEMS + i;
          if (r < n) {
            firsts += (s_flag[r] >> 1) & 1u;
            if (r > 0 && s_ref[r] != s_ref[r - 1]) { ++bnd; m2[1] = r; }
          }
        }
        for (uint32_t v = (uint32_t)tid; v < cnt; v += NT)
          m2[0] = max(m2[0], ((unsigned long long)(s_hpos[v + 1] - s_hpos[v]) << 32) | (0xffffffffu - v));
        uint32_t tot2;
        const uint32_t ex = block_excl_sum<NT>(firsts | (bnd << 16), s_w32, tot2);   // both <= 4096: no carry between the halves
        block_max<NT, 2>(m2, s_w64);
        uint32_t fo = ex & 0xffffu;
        run_before = ex >> 16;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t r = (uint32_t)tid * ITEMS + i;
          if (r < n && (s_flag[r] & 2)) s_fo[s_ref[r]] = (uint16_t)fo++;
        }
        runs = (tot2 >> 16) + 1u;
        last_run = (uint32_t)m2[1];
        max_cnt = cnt ? (uint32_t)(m2[0] >> 32) : 0u;
        const_ref = cnt ? 0xffffffffu - (uint32_t)m2[0] : 0u;
        if (null_cnt > max_cnt) { max_cnt = null_cnt; const_ref = cnt; }   // NULL only when strictly more frequent
        // ---- CONST exceptions: rows whose ref is not the constant's ------------------------------------------------------
        const uint32_t exc = n - max_cnt;
        const bool const_ok = !(exc > 32u || exc > max(n * 10u / 100u, 1u));
        if ((want == OBGPU_ENC_CONST || want == OBGPU_ENC_AUTO) && const_ok && exc > 0) {
          uint32_t ne = 0;
          unsigned long long m1[1] = {0ull};
#pragma unroll
          for (int i = 0; i < ITEMS; ++i) {
            const uint32_t r = (uint32_t)tid * ITEMS + i;
            if (r < n && s_ref[r] != const_ref) { ++ne; m1[0] = r; }
          }
          uint32_t tot3;
          exc_before = block_excl_sum<NT>(ne, s_w32, tot3);
          block_max<NT, 1>(m1, s_w64);
          exc_max_row = (uint32_t)m1[0];
        }
        __syncthreads();   // s_fo
      }
    }

    // ---- choice -------------------------------------------------------------------------------------------------------------
    int use = want;
    if (want == OBGPU_ENC_AUTO) {
      ColFacts f;
      f.n = n; f.null_cnt = null_cnt; f.distinct = cnt; f.max_cnt = max_cnt; f.runs = runs; f.last_run = last_run;
      f.exc_max_row = exc_max_row; f.max_integer = max_integer; f.tmin = tmin; f.tmax = tmax;
      f.ts = (int)ts; f.sc = cs.sc; f.ext_bit = (int)ext_bit; f.enable_bp = enable_bp;
      use = choose_auto(f);
    }
    if (use == OBGPU_ENC_INTEGER_BASE_DIFF && tmax == tmin) use = OBGPU_ENC_RAW;   // zero delta (or no value): written as RAW

    // ---- layout + pack ------------------------------------------------------------------------------------------------------
    uint32_t *h = img32 + (kHeaderSize + 16u * (uint32_t)c) / 4u;   // ObColumnHeader
    const uint32_t off = at;
    uint32_t bytes = 0, attr = 0, length = 0;
    // [ext bits][bit-packed cells] then byte-packed cells (fill_column_store); value(r) of the non-NULL rows
    auto fixed_store = [&](uint32_t base, bool need_ext, bool bp, uint32_t size, auto value_of, bool include_null_cells) {
      const uint32_t ext_bits = need_ext ? ext_bit * n : 0u;
      const uint32_t bits_size = (ext_bits + (bp ? size * n : 0u) + 7u) / 8u;
      const uint32_t w = bp ? size : 8u * size;
      const uint32_t cell0 = bp ? base * 8u + ext_bits : (base + bits_size) * 8u;
      for (uint32_t r = (uint32_t)tid; r < n; r += NT) {
        const bool is_null = has_null && nulls && nulls[r] != 0;
        if (is_null && need_ext) or_bits(img32, base * 8u + r * ext_bit, 1u, 1ull);   // STORED_NULL
        if (!is_null || include_null_cells) or_bits(img32, cell0 + r * w, w, value_of(r));
      }
      return bits_size + (bp ? 0u : size * n);
    };
    auto put = [&](uint32_t byte_at, uint32_t nbytes, unsigned long long x) { or_bits(img32, byte_at * 8u, 8u * nbytes, x); };
    auto dict_value = [&](uint32_t v) { return (s_key[s_hpos[v]] + tmin) ^ sign; };   // sorted dictionary entry v (store image)
    const uint32_t dsz = enable_bp ? int_size_bytes(max_integer) : byte_packed_size(max_integer);
    const uint32_t max_ref = has_null ? cnt : cnt - 1u;

    if (use == OBGPU_ENC_RAW) {
      bool bp;
      const uint32_t size = packing_size(max_integer, enable_bp, bp);
      // ObRawEncoder::traverse (ob_raw_encoder.cpp:106-110,150-155): NULLs dominate -> var-stored column -> the host writer
      host = bp ? (unsigned long long)size * null_cnt > (unsigned long long)n * 16ull : (unsigned long long)size * null_cnt > (unsigned long long)n * 2ull;
      if (!host) {
        attr = 0x1u | (has_null ? 0x2u : 0u) | (bp ? 0x4u : 0u);
        length = size;
        bytes = fixed_store(off, has_null, bp, size, [&](uint32_t r) { return (unsigned long long)vals[r] & cs.store_mask; }, false);
      }
    } else if (use == OBGPU_ENC_INTEGER_BASE_DIFF) {
      bool bp;
      const uint32_t size = packing_size(tmax - tmin, true, bp);
      attr = 0x1u | (bp ? 0x4u : 0u) | (has_null ? 0x2u : 0u);
      length = 2u + ts;
      if (tid == 0) { put(off + 1u, 1u, size); put(off + 2u, ts, tmin ^ sign); }   // IntegerBaseDiffHeader{0, size}, base
      bytes = length + fixed_store(off + length, has_null, bp, size,
                                   [&](uint32_t r) { return (((unsigned long long)vals[r] & cs.store_mask) ^ sign) - tmin; }, false);
    } else if (use == OBGPU_ENC_DICT) {
      host = cnt == 0;   // all-NULL column: the host writer refuses DICT
      if (!host) {
        bool bp;
        const uint32_t size = packing_size(max_ref, enable_bp, bp);
        attr = 0x1u | (bp ? 0x4u : 0u);
        length = 9u + cnt * dsz;
        if (tid == 0) { put(off + 1u, 1u, size); put(off + 2u, 4u, cnt); put(off + 6u, 2u, dsz); put(off + 8u, 1u, 0x3u); }   // FIX_LENGTH | IS_SORTED
        for (uint32_t v = (uint32_t)tid; v < cnt; v += NT) put(off + 9u + v * dsz, dsz, dict_value(v));
        bytes = length + fixed_store(off + length, false, bp, size, [&](uint32_t r) { return (unsigned long long)s_ref[r]; }, true);
      }
    } else if (use == OBGPU_ENC_RLE) {
      host = cnt == 0;
      if (!host) {
        const uint32_t rib = byte_packed_size(last_run), refb = byte_packed_size(max_ref);
        const uint32_t head = 10u + runs * (rib + refb);
        if (tid == 0) {
          put(off + 1u, 1u, (rib & 7u) | ((refb & 7u) << 3)); put(off + 2u, 4u, runs); put(off + 6u, 4u, head);   // RLEMetaHeader
          put(off + head + 2u, 4u, cnt); put(off + head + 6u, 2u, dsz); put(off + head + 8u, 1u, 0x1u);           // unsorted dict meta
        }
        // runs in row order: run k starts at row_id[k] with first-occurrence ref[k]; the rows of a thread are consecutive
        uint32_t k = run_before;
#pragma unroll
        for (int i = 0; i < ITEMS; ++i) {
          const uint32_t r = (uint32_t)tid * ITEMS + i;
          if (r < n && (r == 0 || s_ref[r] != s_ref[r - 1])) {
            const uint32_t ref = s_ref[r], kk = r == 0 ? 0u : ++k;
            put(off + 10u + kk * rib, rib, r);
            put(off + 10u + runs * rib + kk * refb, refb, ref == cnt ? cnt : (uint32_t)s_fo[ref]);
          }
        }
        for (uint32_t v = (uint32_t)tid; v < cnt; v += NT) put(off + head + 9u + s_fo[v] * dsz, dsz, dict_value(v));
        bytes = length = head + 9u + cnt * dsz;
      }
    } else {   // OBGPU_ENC_CONST
      const uint32_t exc = n - max_cnt;
      host = exc > 32u || exc > max(n * 10u / 100u, 1u);
      if (!host) {
        if (exc == 0) {
          if (tid == 0) {
            put(off + 2u, 1u, cnt == 0 ? 1u : 0u); put(off + 4u, 2u, 6u);   // const_ref_ (1: every row NULL), offset_
            if (cnt != 0) put(off + 6u, ts, dict_value(0));
          }
          bytes = 6u + (cnt != 0 ? ts : 0u);
        } else {
          const uint32_t rib = byte_packed_size(exc_max_row), head = 6u + exc * (rib + 1u);
          if (tid == 0) {
            put(off + 1u, 1u, exc); put(off + 2u, 1u, const_ref); put(off + 3u, 1u, rib & 7u); put(off + 4u, 2u, head);
            put(off + head + 2u, 4u, cnt); put(off + head + 6u, 2u, dsz); put(off + head + 8u, 1u, 0x3u);   // sorted dict meta
          }
          uint32_t k = exc_before;
#pragma unroll
          for (int i = 0; i < ITEMS; ++i) {
            const uint32_t r = (uint32_t)tid * ITEMS + i;
            if (r < n && s_ref[r] != const_ref) {
              put(off + 6u + k, 1u, s_ref[r]);
              put(off + 6u + exc + k * rib, rib, r);
              ++k;
            }
          }
          for (uint32_t v = (uint32_t)tid; v < cnt; v += NT) put(off + head + 9u + v * dsz, dsz, dict_value(v));
          bytes = head + 9u + cnt * dsz;
        }
        length = bytes;
      }
    }
    if (!host && tid == 0) {
      h[0] = ((uint32_t)use << 8) | (attr << 16) | ((uint32_t)cs.obj_type << 24);
      h[1] = 0u;
      h[2] = off - meta0;
      h[3] = length;
    }
    at += bytes;
    __syncthreads();   // the scratch of this column is read until here
  }

  const uint32_t size = host ? 0u : at;
  const uint32_t slot = (size + p.align - 1u) & ~(p.align - 1u);
  if (tid == 0 && blk > 0) {   // publish the aligned size for the look-backs of the following blocks
    volatile unsigned long long *flags = p.flags;
    flags[blk] = (1ull << 62) | slot;
  }
  if (size != 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // pack writes -> visible to the bulk copy issued by thread 0
    __syncthreads();
    payload_crc_part<NT>(p, img32, tab, size, s_red, tid, lane, warp);
  }
  if (tid == 0) s_off = look_back(p, blk, size, slot, host);
  __syncthreads();
  if (tid == 0 && size != 0)
    finish_block<NW>(p, smem, tab, s_red, size, slot, n, ext_bit, (uint32_t)min(original, 0x7fffffffull), s_off);
}

}  // namespace enc

template <int ITEMS>
static int enc_launch_codecs(obgpu_ctx *ctx, enc::Params &p, int32_t n_cols, int32_t rowkey_col_cnt, int64_t total_rows, int64_t rows_per_block,
                             int32_t align, int64_t n_blocks64, int64_t slot_cap, obgpu_encoded **out) {
  const size_t smem = (size_t)slot_cap + 4096 + enc::codec_scratch_bytes<ITEMS>(n_cols);
  cudaFuncAttributes fa{};
  cudaError_t err = cudaFuncGetAttributes(&fa, enc::obgpu_encode_codecs_kernel<ITEMS>);
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); return OBGPU_ERR_SYS; }
  if ((int64_t)(smem + fa.sharedSizeBytes) > (int64_t)ctx->max_smem_optin) return OBGPU_NOT_SUPPORTED;
  obgpu_encoded *e = nullptr;
  int rc = enc_alloc(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, &e);
  if (rc != OBGPU_SUCCESS) return rc;
  err = cudaFuncSetAttribute(enc::obgpu_encode_codecs_kernel<ITEMS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); obgpu_encoded_free(e); return OBGPU_ERR_SYS; }
  enc::obgpu_encode_codecs_kernel<ITEMS><<<(unsigned)e->n_blocks, enc::kCodecThreads, smem, ctx->stream>>>(p);
  ctx->launches++;
  err = cudaGetLastError();
  if (err != cudaSuccess) { ctx->err = cudaGetErrorString(err); obgpu_encoded_free(e); return OBGPU_ERR_SYS; }
  *out = e;
  return OBGPU_SUCCESS;
}

extern "C" {

int obgpu_encode_columns_with(obgpu_ctx *ctx, const obgpu_encode_col *cols, const int32_t *encodings, int32_t n_cols, int32_t rowkey_col_cnt,
                              int64_t total_rows, int64_t rows_per_block, int32_t align, obgpu_encoded **out) {
  if (!out) return OBGPU_INVALID_ARGUMENT;
  enc::Params p{};
  int64_t n_blocks64 = 0;
  int rc = enc_prepare(ctx, cols, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, p, n_blocks64);
  if (rc != OBGPU_SUCCESS) return rc;
  bool any_codec = false;
  int64_t bound = (int64_t)enc::kHeaderSize + 16 * n_cols;   // the largest block the requested codecs can write
  for (int c = 0; c < n_cols; ++c) {
    const int32_t e = encodings ? encodings[c] : OBGPU_ENC_RAW;
    if (e != OBGPU_ENC_RAW && e != OBGPU_ENC_DICT && e != OBGPU_ENC_RLE && e != OBGPU_ENC_CONST && e != OBGPU_ENC_INTEGER_BASE_DIFF &&
        e != OBGPU_ENC_AUTO)
      return OBGPU_INVALID_ARGUMENT;
    p.col[c].enc = (uint8_t)e;
    any_codec = any_codec || e != OBGPU_ENC_RAW;
    const int64_t n = rows_per_block, ts = p.col[c].ts;
    const int64_t raw = ts * n + (n + 7) / 8 + 1, base_diff = 2 + ts + raw;
    const int64_t dict = 9 + ts * n + 2 * n, rle = 19 + ts * n + 4 * n, cnst = 6 + 32 * 3 + 9 + 33 * ts;   // refs / row ids <= 2 bytes
    int64_t b = raw;
    if (e == OBGPU_ENC_INTEGER_BASE_DIFF) b = base_diff;
    else if (e == OBGPU_ENC_DICT) b = dict;
    else if (e == OBGPU_ENC_RLE) b = rle;
    else if (e == OBGPU_ENC_CONST) b = cnst;
    else if (e == OBGPU_ENC_AUTO) b = std::max({base_diff, dict, rle, cnst});
    bound += b;
  }
  if (!any_codec) return enc_launch_raw(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, out);
  if (rows_per_block > enc::kCodecMaxRows) return OBGPU_NOT_SUPPORTED;
  const int64_t slot_cap = (bound + align - 1) / align * align;
  cudaSetDevice(ctx->device);
  if (rows_per_block <= enc::kCodecThreads * 2)
    return enc_launch_codecs<2>(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, out);
  if (rows_per_block <= enc::kCodecThreads * 4)
    return enc_launch_codecs<4>(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, out);
  if (rows_per_block <= enc::kCodecThreads * 8)
    return enc_launch_codecs<8>(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, out);
  return enc_launch_codecs<16>(ctx, p, n_cols, rowkey_col_cnt, total_rows, rows_per_block, align, n_blocks64, slot_cap, out);
}

}  // extern "C"
