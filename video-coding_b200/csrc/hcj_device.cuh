// hcj_device.cuh — per-thread building blocks of the kernels, written as __host__ __device__ functions so
// that tests/emul can compile the very same code with g++ and check it against the oracle on the CPU
// before any GPU time is spent.  (The emulation is test infrastructure; the product only ever runs
// these functions inside the CUDA kernels of hcj_kernels.cu.)
#pragma once
#include <stdint.h>

#include "hcj_common.h"

#if defined(__CUDACC__)
#define HCJ_HD __host__ __device__ __forceinline__
#else
#define HCJ_HD inline
#endif

namespace hcjdev {

// ------------------------------------------------------------------------------------------------
// Bit reader over the destuffed entropy-coded bytes of one image.
//
// Semantics of Bitstream_reader.From_string (common/src/bitstream_reader.ml:19-38): MSB first, bits at
// or beyond `end_bits` read as zero.  `pos` is an absolute bit position in the image's entropy buffer.
// ------------------------------------------------------------------------------------------------
HCJ_HD uint32_t bswap32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(x, 0, 0x0123);
#else
  return (x >> 24) | ((x >> 8) & 0xff00u) | ((x << 8) & 0xff0000u) | (x << 24);
#endif
}

// Raw (little-endian, unmasked) word `idx` of the stream, 0 past the end.  Kept separate from
// be_word() so that the value of a look-ahead load is not touched (= waited for) before it is needed.
HCJ_HD uint32_t load_raw_word(const uint32_t *__restrict__ words, uint32_t idx, uint32_t end_bits) {
  if ((idx << 5) >= end_bits) return 0u;
#if defined(__CUDA_ARCH__)
  return __ldg(words + idx);
#else
  return words[idx];
#endif
}
// Big-endian view of a raw word with the bits at or beyond end_bits cleared.
HCJ_HD uint32_t be_word(uint32_t raw, uint32_t idx, uint32_t end_bits) {
  uint32_t w = bswap32(raw);
  const uint32_t bitbase = idx << 5;
  if (bitbase >= end_bits) return 0u;
  const uint32_t rem = end_bits - bitbase;
  if (rem < 32u) w &= ~(0xffffffffu >> rem);
  return w;
}
HCJ_HD uint32_t load_be_word(const uint32_t *__restrict__ words, uint32_t idx, uint32_t end_bits) {
  return be_word(load_raw_word(words, idx, end_bits), idx, end_bits);
}

struct BitReader {
  const uint32_t *words;
  uint32_t end_bits;
  uint32_t pos;
  uint32_t widx;
  uint32_t w0, w1;  // big-endian words widx, widx + 1: the 32-bit window lives in these
  uint32_t wn_raw;  // raw word widx + 2, requested one refill ahead so that its latency is never waited for

  HCJ_HD void init(const uint32_t *words_, uint32_t pos_, uint32_t end_bits_) {
    words = words_;
    end_bits = end_bits_;
    pos = pos_;
    widx = pos_ >> 5;
    w0 = load_be_word(words, widx, end_bits);
    w1 = load_be_word(words, widx + 1, end_bits);
    wn_raw = load_raw_word(words, widx + 2, end_bits);
  }
  // The next 32 bits, MSB-aligned.
  HCJ_HD uint32_t window() const {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(w1, w0, pos);
#else
    uint32_t s = pos & 31u;
    return s ? (w0 << s) | (w1 >> (32u - s)) : w0;
#endif
  }
  // Advance by n <= 32 bits.
  HCJ_HD void skip(uint32_t n) {
    pos += n;
    uint32_t nidx = pos >> 5;
    if (nidx != widx) {
      widx = nidx;
      w0 = w1;
      w1 = be_word(wn_raw, nidx + 1, end_bits);
      wn_raw = load_raw_word(words, nidx + 2, end_bits);
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Huffman tables as the kernels see them: one 32-bit "fast" entry per HCJ_LUT_BITS-bit prefix, byte
// aligned so that each field is one PRMT away:
//   [7:0] code length + magnitude bits, [15:8] code length, [23:16] 32 - size,
//   [31:24] zig-zag advance: run + 1 (1..16); HCJ_ZADV_EOB for end-of-block; 1 for a DC symbol;
//   bit 31 = not resolved by the prefix: a longer code (sub-table in shared memory, or the model's full
//   2^max_bits table in global memory for pathological tables); HCJ_FAST_NONE = no such code.
// Adding the advance to the zig-zag index z (1..63) classifies the symbol with no further test:
//   < 64 more coefficients follow; == 64 coefficient 63 was the last; 65..79 the run went past
//   coefficient 63 (the model raises); [HCJ_ZADV_EOB + 1, HCJ_ZADV_EOB + 63] end of block; >= 256 no code.
// ------------------------------------------------------------------------------------------------
#define HCJ_FAST_SLOW 0x80000000u
#define HCJ_FAST_SUB (1u << 8)   // slow entry: look in sub-table (entry & 7)
#define HCJ_FAST_FULL (2u << 8)  // slow entry: look in the full table (global memory)
#define HCJ_ZADV_EOB 96u
#define HCJ_FAST_NONE 0xff200000u  // advance 255, size 0, consumes no bits

// (length << 8 | data) of Tables.Lut -> fast entry.
HCJ_HD uint32_t fast_entry(uint32_t e16, bool isdc) {
  const uint32_t len = e16 >> 8, data = e16 & 0xffu;
  const uint32_t size = isdc ? data : data & 15u;
  const uint32_t zadv = isdc ? 1u : (data == 0u ? HCJ_ZADV_EOB : (data >> 4) + 1u);
  return (len + size) | (len << 8) | ((32u - size) << 16) | (zadv << 24);
}
// Primary-table entry (hcj_common.h) -> fast entry.
HCJ_HD uint32_t fast_entry_from_primary(uint32_t p16, uint32_t max_bits, bool isdc) {
  if (p16 & 0x8000u) return HCJ_FAST_SLOW | HCJ_FAST_SUB | (p16 & (HCJ_LUT_NSUB - 1));
  if (p16 == 0u) return max_bits > HCJ_LUT_BITS ? (HCJ_FAST_SLOW | HCJ_FAST_FULL) : HCJ_FAST_NONE;
  return fast_entry(p16, isdc);
}
// Sub-table / full-table entry -> fast entry.
HCJ_HD uint32_t fast_entry_or_none(uint32_t e16, bool isdc) { return e16 ? fast_entry(e16, isdc) : HCJ_FAST_NONE; }

HCJ_HD uint32_t shr_clamp(uint32_t x, uint32_t n) {  // x >> n with n in [0, 32]
#if defined(__CUDA_ARCH__)
  uint32_t r;
  asm("shr.b32 %0, %1, %2;" : "=r"(r) : "r"(x), "r"(n));
  return r;
#else
  return n >= 32u ? 0u : x >> n;
#endif
}
HCJ_HD uint32_t byte_of(uint32_t x, int k) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(x, 0, 0x4440 | k);
#else
  return (x >> (8 * k)) & 0xffu;
#endif
}

// The tables of the CTA's image as the fast loops see them (pointers into shared memory in the kernels;
// built in the kernel body and passed by value so that the loads compile to LDS).  A table is named by
// the offset of its fast entries: toff = (pair * 2 + (0 = dc, 1 = ac)) * HCJ_LUT_SIZE.
struct alignas(16) BlkInfo {
  uint32_t tdc, tac, qoff;  // dc toff, ac toff, quant offset (entries)
  uint32_t comp_qmax;       // scan component | largest AC quant entry << 8
};
struct FastTables {
  const uint32_t *fast;         // [table][HCJ_LUT_SIZE]
  const uint32_t *sub;          // [table][HCJ_LUT_NSUB * HCJ_LUT_SUB_SIZE], fast entries
  const uint32_t *max_bits;     // [table]
  const uint16_t *const *full;  // [table] -> global memory, (length << 8) | data
  const BlkInfo *blkinfo;       // [block-in-MCU]
  const int32_t *quant;         // [scan component][128]
  const uint32_t *multi;        // [pair][HCJ_LUT_SIZE] multi-symbol AC entries of the synchronisation passes (or null)
};

// `e` has HCJ_FAST_SLOW set.  Returns a resolved entry or HCJ_FAST_NONE.  The sub-tables are kept in a uniform shape
// (load_tables): HCJ_LUT_SUB_SIZE entries each, indexed by the HCJ_LUT_SUB_BITS bits that follow the primary index,
// whatever the table's longest code.
HCJ_HD uint32_t fast_lookup_slow(const FastTables &T, uint32_t toff, uint32_t e, uint32_t win, bool isdc) {
  if (e == HCJ_FAST_NONE) return e;
  const uint32_t ti = toff >> HCJ_LUT_BITS;
  if (e & HCJ_FAST_SUB)
    return T.sub[ti * (HCJ_LUT_NSUB * HCJ_LUT_SUB_SIZE) + (e & (HCJ_LUT_NSUB - 1)) * HCJ_LUT_SUB_SIZE +
                 ((win >> (32 - HCJ_LUT_BITS - HCJ_LUT_SUB_BITS)) & (HCJ_LUT_SUB_SIZE - 1))];
  return fast_entry_or_none(T.full[ti][win >> (32u - T.max_bits[ti])], isdc);
}
// Entry `i` of a uniform sub-table from the host's (a verbatim slice of the full table: 2^(max_bits - HCJ_LUT_BITS)
// entries, indexed by the bits between the primary index and the longest code).
HCJ_HD uint32_t sub_source_index(uint32_t i, uint32_t max_bits) {
  const uint32_t have = max_bits > (uint32_t)HCJ_LUT_BITS ? max_bits - (uint32_t)HCJ_LUT_BITS : 0u;
  return have >= (uint32_t)HCJ_LUT_SUB_BITS ? i : i >> ((uint32_t)HCJ_LUT_SUB_BITS - have);
}
HCJ_HD uint32_t fast_lookup(const FastTables &T, uint32_t toff, uint32_t win, bool isdc) {
  uint32_t e = T.fast[toff + (win >> (32 - HCJ_LUT_BITS))];
  if (e & HCJ_FAST_SLOW) e = fast_lookup_slow(T, toff, e, win, isdc);
  return e;
}

// fast entry -> (length << 8) | data of Tables.Lut (decoder.ml:89-105); lossless
HCJ_HD uint32_t fast_to_e16(uint32_t e, bool isdc) {
  const uint32_t len = (e >> 8) & 0xffu, size = 32u - ((e >> 16) & 0xffu), zadv = e >> 24;
  return (len << 8) | (isdc ? size : zadv == HCJ_ZADV_EOB ? 0u : ((zadv - 1u) << 4) | size);
}

// Huffman tables of one scan component as the literal decode loops see them.
struct Tables {
  uint32_t dc_off, ac_off;  // toff of the component's tables in FastTables
  uint32_t dc_max_bits, ac_max_bits;
};

// The hot lookup tables of the CTA's image.  In the kernels these point into __shared__ arrays and the
// struct is built in the kernel body and passed by value, so that after inlining the compiler knows
// the address space and emits LDS (a generic load costs a long-scoreboard round trip per symbol).
struct Local {
  FastTables ft;
  const int32_t *quant;     // [scan component][128]: 64 plain entries + 64 in dp2a form
  const uint8_t *blk_comp;  // [bpm] block-in-MCU -> scan component
};

// Tables.Lut lookup (decoder.ml:89-105): (length << 8) | data, 0 = None.
HCJ_HD uint32_t lut_lookup(const Local &L, uint32_t toff, bool isdc, uint32_t win) {
  const uint32_t e = fast_lookup(L.ft, toff, win, isdc);
  return (e & HCJ_FAST_SLOW) ? 0u : fast_to_e16(e, isdc);
}

// Decoder.mag' (decoder.ml:73-79) for cat >= 1 on the cat bits that follow the code.
HCJ_HD int32_t extend(uint32_t bits, uint32_t cat) {
  int32_t v = (int32_t)bits;
  return (bits >> (cat - 1u)) ? v : v - (int32_t)(1u << cat) + 1;
}

// Clears one 128-byte coefficient block (clear_block, decoder.ml:112-116) with full-sector stores.  Done
// by the thread that begins the block right before its first coefficient store: the sector is then
// resident (dirty) in L2 when the scattered 2-byte stores arrive, so they neither fetch the line from HBM
// nor need a separate clearing pass over the whole coefficient buffer.
HCJ_HD void zero_block(int16_t *blk) {
#if defined(__CUDA_ARCH__)
  uint4 *p = reinterpret_cast<uint4 *>(blk);
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
  for (int j = 0; j < 8; j++) p[j] = z;
#else
  for (int j = 0; j < 64; j++) blk[j] = 0;
#endif
}

// ------------------------------------------------------------------------------------------------
// Exact decode of one 8x8 block (Decoder.huffman_decode, decoder.ml:118-140) into a zero-initialised
// int16 block (cleared here) in zig-zag order; slot 0 receives the RESOLVED dc (pred + diff, decoder.ml:143).
// `seg_bits` is the length of the reader the model would be using (for the `show` bound, reader.ml:32).
// Returns 0 or the status of the exception the model raises.
// ------------------------------------------------------------------------------------------------
HCJ_HD int decode_block_exact(BitReader &br, const Local L, const Tables &t, uint32_t seg_bits, int32_t &dc_pred,
                              int16_t *__restrict__ blk) {
  zero_block(blk);
  const bool careful = seg_bits <= 16u;
  if (careful && t.dc_max_bits >= seg_bits) return HCJ_DEV_BITS_OOB;
  uint32_t win = br.window();
  uint32_t e = lut_lookup(L, t.dc_off, true, win);
  if (e == 0u) return HCJ_DEV_NO_DC_CODE;
  uint32_t len = e >> 8, cat = e & 0xffu;
  int32_t diff = 0;
  if (cat) {
    if (careful && cat >= seg_bits) return HCJ_DEV_BITS_OOB;
    diff = extend((win << len) >> (32u - cat), cat);
  }
  br.skip(len + cat);
  dc_pred += diff;
  if (dc_pred < -32768 || dc_pred > 32767) return HCJ_DEV_DC_RANGE;
  blk[0] = (int16_t)dc_pred;
  uint32_t k = 1;
  while (k < 64u) {
    if (careful && t.ac_max_bits >= seg_bits) return HCJ_DEV_BITS_OOB;
    win = br.window();
    e = lut_lookup(L, t.ac_off, false, win);
    if (e == 0u) return HCJ_DEV_NO_AC_CODE;
    len = e >> 8;
    uint32_t rs = e & 0xffu, size = rs & 15u;
    if (careful && size >= seg_bits && size) return HCJ_DEV_BITS_OOB;
    uint32_t mbits = size ? (win << len) >> (32u - size) : 0u;
    br.skip(len + size);
    if (rs == 0u) break;  // (run, size) = (0, 0): end of block (decoder.ml:131-132)
    k += rs >> 4;
    if (k >= 64u) return HCJ_DEV_COEF_INDEX;
    if (size) blk[k] = (int16_t)extend(mbits, size);  // size 0 (e.g. ZRL) stores 0: already there
    k++;
  }
  return HCJ_DEV_OK;
}

// ------------------------------------------------------------------------------------------------
// Self-synchronising subsequence decode (no restart markers).
//
// The scan is cut into subsequences of S bits.  A decoder state between symbols is (p, c, z):
// bit position, block-in-MCU index, next zig-zag index (0 = a DC symbol comes next).  `sync` decodes
// the symbols that START inside [p, hi) without storing coefficients and reports the state at the
// first symbol start >= hi together with what the final pass needs for its prefix sums: the number of
// blocks begun and the sum of DC differentials per scan component.  On undefined codes / overlong runs
// (only possible while speculating from a wrong state, or in a corrupt stream) it recovers
// deterministically: skip one bit / close the block.  The final pass reports those as errors.
// ------------------------------------------------------------------------------------------------
struct ScanCtx {
  const uint32_t *words;       // destuffed bytes of the image (16-byte aligned)
  uint32_t total_bits;         // 8 * destuffed length
  uint32_t bpm;                // blocks per MCU
  Tables tab[HCJ_MAX_COMP];    // per scan component
  uint32_t *wide_flags;        // bit (blk_base + blk): the block needs the 64-bit IDCT (see HCJ_IDCT_L1_LIMIT)
  uint64_t blk_base;           // index of the image's first block in the batch
};

// A block is decoded by one thread from its DC symbol to its end, which forms the block's sum(|dequantised
// coefficient|) and flags the block when it reaches the limit.
#define HCJ_IDCT_L1_LIMIT_VALUE 60000
#define HCJ_WIDE_SHARE HCJ_IDCT_L1_LIMIT_VALUE

HCJ_HD void flag_wide_block(const ScanCtx &sc, int64_t blk) {
  uint64_t g = sc.blk_base + (uint64_t)blk;
#if defined(__CUDA_ARCH__)
  atomicOr(sc.wide_flags + (g >> 5), 1u << (g & 31u));
#else
  sc.wide_flags[g >> 5] |= 1u << (g & 31u);
#endif
}

struct SubResult {
  uint32_t p, cz;     // end state: cz = (c << 8) | z
  uint32_t nstart;    // DC symbols (blocks begun) decoded
  int32_t dcsum[HCJ_MAX_COMP];
  // The first MCU that begins here (DC symbol of block-in-MCU 0): its position (0xffffffff: none) and how many
  // blocks were begun before it; the DC sums up to it go to the `dpre` argument of the decode functions.
  uint32_t first_p, nbefore;
};

// One symbol, DC or AC, decoded with the same instruction stream (lanes of a warp are rarely all in the
// same phase, so separate DC / AC branches would both be executed on almost every iteration).
struct Symbol {
  uint32_t e;      // LUT entry, 0 = undefined code
  uint32_t nbits;  // code length + magnitude bits
  uint32_t run, size;
  int32_t value;   // extended magnitude (0 when size == 0)
};

HCJ_HD Symbol read_symbol(const BitReader &br, const Local L, const Tables &t, bool isdc) {
  Symbol s;
  const uint32_t win = br.window();
  const uint32_t e = lut_lookup(L, isdc ? t.dc_off : t.ac_off, isdc, win);
  const uint32_t len = e >> 8, rs = e & 0xffu;
  s.e = e;
  s.size = isdc ? rs : rs & 15u;
  s.run = isdc ? 0u : rs >> 4;
  s.nbits = len + s.size;
  const uint32_t mbits = s.size ? (win << len) >> (32u - s.size) : 0u;
  s.value = s.size ? extend(mbits, s.size) : 0;
  return s;
}

HCJ_HD void subseq_sync(const ScanCtx &sc, const Local L, uint32_t p, uint32_t cz, uint32_t hi, SubResult &r, uint32_t end_bits,
                        int32_t *dpre /* [HCJ_MAX_COMP], written when the first MCU start is met */) {
  uint32_t c = cz >> 8, z = cz & 0xffu;
  uint32_t nstart = 0;
  int32_t d0 = 0, d1 = 0, d2 = 0, d3 = 0;
  BitReader br;
  br.init(sc.words, p, end_bits);  // end of the scan / of the restart interval: bits beyond it read as zero
  uint32_t comp = L.blk_comp[c];
  Tables t = sc.tab[comp];
  r.first_p = 0xffffffffu;
  r.nbefore = 0;
  while (br.pos < hi) {
    const bool isdc = z == 0u;
    const Symbol s = read_symbol(br, L, t, isdc);
    // The first MCU start is where its DC symbol is LOOKED FOR: if the code there is undefined, the exact pass of the
    // thread that starts here raises what the model raises (found by the soak: the position used to be recorded after
    // the skipped bits, and the error was lost).
    if (isdc && c == 0u && r.first_p == 0xffffffffu) {
      r.first_p = br.pos, r.nbefore = nstart;
      dpre[0] = d0, dpre[1] = d1, dpre[2] = d2, dpre[3] = d3;
    }
    if (s.e == 0u) {  // undefined code: resynchronise one bit later
      br.skip(1);
      continue;
    }
    br.skip(s.nbits);
    const int32_t diff = isdc ? s.value : 0;
    d0 += comp == 0u ? diff : 0;
    d1 += comp == 1u ? diff : 0;
    d2 += comp == 2u ? diff : 0;
    d3 += comp == 3u ? diff : 0;
    nstart += isdc ? 1u : 0u;
    // next zig-zag index: 1 after a DC; 64 on EOB; past 63 closes the block too (coefficient 63, or an
    // overlong run met while speculating)
    z = isdc ? 1u : ((s.e & 0xffu) ? z + s.run + 1u : 64u);
    if (z >= 64u) {
      z = 0;
      c = c + 1u == sc.bpm ? 0u : c + 1u;
      comp = L.blk_comp[c];
      t = sc.tab[comp];
    }
  }
  r.p = br.pos;
  r.cz = (c << 8) | z;
  r.nstart = nstart;
  r.dcsum[0] = d0;
  r.dcsum[1] = d1;
  r.dcsum[2] = d2;
  r.dcsum[3] = d3;
}

// Final pass of one thread: a run of whole MCUs.  It starts at an MCU boundary (p, block-in-MCU c = 0, DC next) with
// the DC predictors `pred`; `blk` is the index (within the image) of the block before the first one it decodes.  It
// decodes the MCUs (blocks < `nblocks`) that BEGIN before `hi` (the one in progress at `hi` is finished: the thread of
// the next subsequence starts at the first MCU that begins in its own bits - so the lanes of a warp, which run in lock
// step block by block, are all in the same block-in-MCU, luma with luma and chroma with chroma) or at / beyond
// `end_bits` (nobody else's: the model's reader delivers zero bits there and the unit's blocks are decoded whatever
// the bits say); with hi >= end_bits it runs until block nblocks - 1 is complete.  Stores
// coefficients (zig-zag, DC resolved) into `coefs`; every block is cleared right before its DC store.
HCJ_HD int subseq_write(const ScanCtx &sc, const Local L, uint32_t p, uint32_t c, uint32_t hi, uint32_t end_bits, int64_t blk,
                        int32_t pred[HCJ_MAX_COMP], int64_t nblocks, int16_t *__restrict__ coefs, uint32_t *err_pos,
                        uint32_t z = 0, uint32_t share0 = 0) {
  BitReader br;
  br.init(sc.words, p, end_bits);
  uint32_t comp = L.blk_comp[c];
  Tables t = sc.tab[comp];
  const int32_t *q = L.quant + comp * 128;
  int32_t p0 = pred[0], p1 = pred[1], p2 = pred[2], p3 = pred[3];
  int16_t *out = coefs + blk * 64;
  uint32_t share = share0;  // sum(|dequantised coefficient|) of the block in progress
  int err = HCJ_DEV_OK;
  for (;;) {
    const bool isdc = z == 0u;
    if (isdc && (blk + 1 >= nblocks || (c == 0u && br.pos >= hi && br.pos < end_bits))) break;  // every block is complete / the next MCU is not this thread's
    const Symbol s = read_symbol(br, L, t, isdc);
    if (s.e == 0u) {
      err = isdc ? HCJ_DEV_NO_DC_CODE : HCJ_DEV_NO_AC_CODE;
      break;
    }
    br.skip(s.nbits);
    const bool eob = !isdc && (s.e & 0xffu) == 0u;
    const uint32_t zi = isdc ? 0u : z + s.run;  // where this symbol's value goes
    if (zi >= 64u && !eob) {
      err = HCJ_DEV_COEF_INDEX;
      break;
    }
    int32_t v = s.value;
    if (isdc) {
      const int32_t pv = (comp == 0u ? p0 : comp == 1u ? p1 : comp == 2u ? p2 : p3) + v;
      p0 = comp == 0u ? pv : p0;
      p1 = comp == 1u ? pv : p1;
      p2 = comp == 2u ? pv : p2;
      p3 = comp == 3u ? pv : p3;
      v = pv;
      if (pv < -32768 || pv > 32767) {
        err = HCJ_DEV_DC_RANGE;
        break;
      }
      blk++;
      out += 64;
      zero_block(out);
    }
    if (isdc || (s.size != 0u && !eob)) {
      out[zi] = (int16_t)v;
      share += (uint32_t)(v < 0 ? -v : v) * (uint32_t)q[zi];
    }
    z = eob ? 64u : zi + 1u;
    if (z >= 64u) {
      if (share >= (uint32_t)HCJ_IDCT_L1_LIMIT_VALUE) flag_wide_block(sc, blk);
      share = 0;
      z = 0;
      c = c + 1u == sc.bpm ? 0u : c + 1u;
      comp = L.blk_comp[c];
      t = sc.tab[comp];
      q = L.quant + comp * 128;
    }
  }
  if (err) *err_pos = br.pos;
  return err;
}

// ================================================================================================
// Fast symbol loops (shared by K2 and K3).
//
// The loops above are the literal ones: every model exception, the zero-extending reader and the `show`
// bound are in them, and their many data-dependent branches leave less than half of a warp's lanes
// active.  The fast steps below decode the same symbols with straight-line code:
//   * one 32-bit table entry per symbol carries everything the step needs (FastTables above);
//   * the reader keeps four words in registers (two of them still raw: their loads were issued two
//     refills ago) and never masks: a lane leaves the fast loop 32 bits before the end of its data;
//   * a step tests nothing: what happened is read off the zig-zag index afterwards (see the table
//     format), by the code that runs once per block, not once per symbol;
//   * errors are not decided here: a lane that meets an undefined code or a DC out of int16 stops BEFORE
//     that symbol with its state intact and the literal loop carries on from there and raises what the
//     model raises; a run past coefficient 63 is the one error reported directly (same status and
//     position as the literal loop: it too has consumed the symbol when it raises).
// ================================================================================================
// Unmasked reader: words pos/32 .. pos/32 + 3 in registers.  Only valid while pos + 32 <= end of data.
struct FastReader {
  const uint32_t *words;
  uint32_t pos, w0, w1, r0, r1;
  HCJ_HD static uint32_t ld(const uint32_t *p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
  }
  HCJ_HD void init(const uint32_t *words_, uint32_t pos_) {
    words = words_;
    pos = pos_;
    const uint32_t i = pos_ >> 5;
    w0 = bswap32(ld(words + i));
    w1 = bswap32(ld(words + i + 1));
    r0 = ld(words + i + 2);
    r1 = ld(words + i + 3);
  }
  HCJ_HD uint32_t window() const {
#if defined(__CUDA_ARCH__)
    return __funnelshift_l(w1, w0, pos);
#else
    uint32_t s = pos & 31u;
    return s ? (w0 << s) | (w1 >> (32u - s)) : w0;
#endif
  }
  HCJ_HD void consume(uint32_t n) {  // n < 32
    const uint32_t np = pos + n;
    const uint32_t cross = (np ^ pos) & 32u;
    pos = np;
    if (cross) {
      w0 = w1;
      w1 = bswap32(r0);
      r0 = r1;
    }
#if defined(__CUDA_ARCH__)
    // The load writes r1 in place (no temporary + move, which would wait for the data right here): its
    // value is first looked at two refills from now.  (Scoreboards are per warp, so the lane that refills in
    // the next step does wait for this load: L2::128B makes that an L2 hit for 31 words out of 32.)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %2, 0;\n\t@p ld.global.nc.L2::128B.u32 %0, [%1];\n\t}"
        : "+r"(r1)
        : "l"(words + (np >> 5) + 3), "r"(cross));
#else
    if (cross) r1 = ld(words + (np >> 5) + 3);
#endif
  }
};

// value of the `size` magnitude bits that follow a code of `len` bits (Decoder.mag', decoder.ml:73-79);
// sh = 32 - size; 0 when size == 0
HCJ_HD int32_t fast_value(uint32_t win, uint32_t len, uint32_t sh) {
  const uint32_t t = win << len;
  const uint32_t m = shr_clamp(t, sh), mask = shr_clamp(0xffffffffu, sh);
  return (int32_t)m - (int32_t)(mask & ~(uint32_t)((int32_t)t >> 31));
}

// What a zig-zag index says after an AC step (z was 1..63 before it).
HCJ_HD bool z_block_done(uint32_t z) { return z >= 64u; }
HCJ_HD bool z_overrun(uint32_t z) { return z > 64u && z <= HCJ_ZADV_EOB; }  // run past coefficient 63
HCJ_HD bool z_no_code(uint32_t z) { return z >= 256u; }

// ---- exact pass -------------------------------------------------------------------------------
struct ExactLane {
  FastReader br;
  uint32_t c, z;            // block-in-MCU; next zig-zag index (0 = at a block boundary)
  uint32_t tdc, tac, qoff;  // tables of the current scan component
  uint32_t comp;
  int32_t blk;              // block in progress (at a boundary: the last one begun)
  int32_t pcur, p0, p1, p2, p3;
  // Wide-block guard (HCJ_WIDE_SHARE): `share` = exact sum(|coef| * q) of what the lane knows exactly (the
  // DC it decoded, what a previous pass handed over); the AC symbols of the fast steps only add |coef| to
  // `sumabs` (no table load per symbol): share + sumabs * qmax bounds the lane's share from above, and only
  // when that bound reaches the limit is the exact value formed from the staged row (exact_share).
  uint32_t share, sumabs, qmax;
};

HCJ_HD void exact_bind_block(ExactLane &s, const FastTables T) {  // tables and predictor of block-in-MCU s.c
  const BlkInfo bi = T.blkinfo[s.c];
  s.tdc = bi.tdc;
  s.tac = bi.tac;
  s.qoff = bi.qoff;
  s.comp = bi.comp_qmax & 0xffu;
  s.qmax = bi.comp_qmax >> 8;
  s.pcur = s.comp == 0u ? s.p0 : s.comp == 1u ? s.p1 : s.comp == 2u ? s.p2 : s.p3;
}
HCJ_HD void exact_save_pred(ExactLane &s) {
  s.p0 = s.comp == 0u ? s.pcur : s.p0;
  s.p1 = s.comp == 1u ? s.pcur : s.p1;
  s.p2 = s.comp == 2u ? s.pcur : s.p2;
  s.p3 = s.comp == 3u ? s.pcur : s.p3;
}
// after a completed block: on to the next block-in-MCU
HCJ_HD void exact_next_block(ExactLane &s, const FastTables T, uint32_t bpm) {
  exact_save_pred(s);
  s.c = s.c + 1u == bpm ? 0u : s.c + 1u;
  s.z = 0u;
  s.share = 0u;
  s.sumabs = 0u;
  exact_bind_block(s, T);
}
// The lane's exact share of the block in progress; `row` holds the AC coefficients behind `sumabs`.
HCJ_HD bool exact_share_may_be_wide(const ExactLane &s) {
  return s.sumabs >= 0x10000u || (uint64_t)s.share + (uint64_t)s.sumabs * s.qmax >= (uint64_t)HCJ_WIDE_SHARE;
}
HCJ_HD uint32_t exact_share(const ExactLane &s, const FastTables T, const int16_t *row) {
  uint64_t a = s.share;
  for (int zi = 1; zi < 64; zi++) {
    const int32_t v = row[zi];
    a += (uint64_t)(uint32_t)(v < 0 ? -v : v) * (uint32_t)T.quant[s.qoff + zi];
  }
  return a > 0xffffffffull ? 0xffffffffu : (uint32_t)a;
}

// One AC symbol of the block in progress (s.z in 1..63); `row` = the lane's staged block (64 int16,
// zig-zag).  Afterwards s.z tells what happened (z_block_done / z_overrun / z_no_code); an undefined code
// consumes nothing and stores nothing.
HCJ_HD void exact_ac_step(ExactLane &s, const FastTables T, int16_t *row) {
  const uint32_t win = s.br.window();
  const uint32_t e = fast_lookup(T, s.tac, win, false);
  const uint32_t znext = s.z + (e >> 24);
  const uint32_t sh = byte_of(e, 2);
  const int32_t v = fast_value(win, byte_of(e, 1), sh);
  if (sh != 32u && znext <= 64u) {
    row[znext - 1u] = (int16_t)v;
    s.sumabs += (uint32_t)(v < 0 ? -v : v);
  }
  s.br.consume(byte_of(e, 0));
  s.z = znext;
}
// undo the only effect of a step that met an undefined code
HCJ_HD void exact_ac_undo_no_code(ExactLane &s) { s.z -= 255u; }

// The DC symbol that begins the next block (s.z == 0, tables bound).  Returns false, with the state
// untouched, if the literal loop has to look at it (undefined code, predictor out of int16).
HCJ_HD bool exact_dc_step(ExactLane &s, const FastTables T, int16_t *row) {
  const uint32_t win = s.br.window();
  const uint32_t e = fast_lookup(T, s.tdc, win, true);
  const int32_t pc = s.pcur + fast_value(win, byte_of(e, 1), byte_of(e, 2));
  if (e == HCJ_FAST_NONE || pc < -32768 || pc > 32767) return false;
  s.pcur = pc;
  s.blk++;
  row[0] = (int16_t)pc;
  s.share = (uint32_t)(pc < 0 ? -pc : pc) * (uint32_t)T.quant[s.qoff];
  s.sumabs = 0u;
  s.br.consume(byte_of(e, 0));
  s.z = 1u;
  return true;
}

// ---- synchronisation pass (no coefficients): same symbols, only the state and the prefix-sum inputs
//
// The values of AC coefficients do not matter here, so one look-up may swallow SEVERAL AC symbols: entry `idx` of a
// table's multi-symbol form describes the longest run of symbols whose codes lie wholly inside the HCJ_LUT_BITS
// index bits (the magnitude bits of the last one may reach beyond them), ending early after an end-of-block (the next
// symbol is a DC one, other table) and never longer than 31 bits:
//   [7:0] bits consumed by all of them, [15:8] `pre` = zig-zag advance of all but the last, [31:24] total advance
//   (capped at 127: any total that takes z to 64 or beyond closes the block, exactly as a single step would).
// The run is valid for a lane at zig-zag index z iff z + pre < 64 (no symbol before the last one closes the block)
// and every symbol of it starts before the lane's limit; otherwise the lane takes the single-symbol step.  Entries
// whose first code is not resolved by the index bits are copied from the single-symbol table (HCJ_FAST_SLOW set).
HCJ_HD uint32_t multi_sync_entry(const uint32_t *fast_ac /* the table's HCJ_LUT_SIZE single-symbol entries */, uint32_t idx) {
  const uint32_t e = fast_ac[idx];
  if (e & HCJ_FAST_SLOW) return e;
  uint32_t pos = e & 0xffu, pre = 0, adv = e >> 24;
  while (adv != HCJ_ZADV_EOB && pos < (uint32_t)HCJ_LUT_BITS && pre + adv < 63u) {
    const uint32_t e2 = fast_ac[(idx << pos) & (HCJ_LUT_SIZE - 1)];
    if (e2 & HCJ_FAST_SLOW) break;
    if (pos + ((e2 >> 8) & 0xffu) > (uint32_t)HCJ_LUT_BITS) break;  // the code needs bits the index does not have
    if (pos + (e2 & 0xffu) > 31u) break;
    pre += adv;
    adv = e2 >> 24;
    pos += e2 & 0xffu;
  }
  const uint32_t tot = pre + adv > 127u ? 127u : pre + adv;
  return pos | (pre << 8) | (tot << 24);
}

struct SyncLane {
  FastReader br;
  uint32_t c, z;
  uint32_t tdc, tac, comp;
  uint32_t nstart;
  int32_t d0, d1, d2, d3;
  uint32_t first_p, nbefore;  // the first MCU begun (SubResult)
};
HCJ_HD void sync_bind_block(SyncLane &s, const FastTables T) {
  const BlkInfo bi = T.blkinfo[s.c];
  s.tdc = bi.tdc;
  s.tac = bi.tac;
  s.comp = bi.comp_qmax & 0xffu;
}
HCJ_HD void sync_next_block(SyncLane &s, const FastTables T, uint32_t bpm) {
  s.c = s.c + 1u == bpm ? 0u : s.c + 1u;
  s.z = 0u;
  sync_bind_block(s, T);
}
// One look-up: as many AC symbols as the multi-symbol entry holds, or one (see multi_sync_entry).  `lim_m`: a run
// may be taken while the position is below it (= all its symbols start before the end of the subsequence).  An
// undefined code is skipped one bit at a time, as subseq_sync does.  Any s.z >= 64 afterwards closes the block,
// overlong runs included, exactly as in subseq_sync.
HCJ_HD void sync_ac_step_multi(SyncLane &s, const FastTables T, uint32_t lim_m) {
  const uint32_t win = s.br.window();
  const uint32_t idx = win >> (32 - HCJ_LUT_BITS);
  uint32_t e = T.multi[((s.tac - HCJ_LUT_SIZE) >> 1) + idx];
  if (s.z + byte_of(e, 1) >= 64u || s.br.pos >= lim_m) e = T.fast[s.tac + idx];  // the single-symbol entry
  if (e & HCJ_FAST_SLOW) {
    e = fast_lookup_slow(T, s.tac, e, win, false);
    if (e == HCJ_FAST_NONE) e = 1u;  // consume one bit, no advance
  }
  s.br.consume(byte_of(e, 0));
  s.z += e >> 24;
}
// The same, one symbol per look-up (kernels that do not keep the multi-symbol tables).
HCJ_HD void sync_ac_step_single(SyncLane &s, const FastTables T) {
  const uint32_t win = s.br.window();
  uint32_t e = T.fast[s.tac + (win >> (32 - HCJ_LUT_BITS))];
  if (e & HCJ_FAST_SLOW) {
    e = fast_lookup_slow(T, s.tac, e, win, false);
    if (e == HCJ_FAST_NONE) e = 1u;  // consume one bit, no advance
  }
  s.br.consume(byte_of(e, 0));
  s.z += e >> 24;
}
// The DC symbol that begins the next block (s.z == 0, tables bound); an undefined code is skipped one bit at a time.
// The first MCU start met is recorded, with the DC sums up to it in `dpre` (int32 [HCJ_MAX_COMP]).
HCJ_HD void sync_dc_step(SyncLane &s, const FastTables T, int32_t *dpre) {
  const uint32_t win = s.br.window();
  const uint32_t e = fast_lookup(T, s.tdc, win, true);
  if (s.c == 0u && s.first_p == 0xffffffffu) {  // (where the DC symbol is looked for, defined or not: see subseq_sync)
    s.first_p = s.br.pos, s.nbefore = s.nstart;
    dpre[0] = s.d0, dpre[1] = s.d1, dpre[2] = s.d2, dpre[3] = s.d3;
  }
  if (e == HCJ_FAST_NONE) {
    s.br.consume(1u);
    return;
  }
  const int32_t v = fast_value(win, byte_of(e, 1), byte_of(e, 2));
  s.d0 += s.comp == 0u ? v : 0;
  s.d1 += s.comp == 1u ? v : 0;
  s.d2 += s.comp == 2u ? v : 0;
  s.d3 += s.comp == 3u ? v : 0;
  s.nstart++;
  s.br.consume(byte_of(e, 0));
  s.z = 1u;
}

// ------------------------------------------------------------------------------------------------
// Dct.Chen.inverse_8x8 (dct.ml:11-107), bit-exact.
//
// T = int32_t: every value is held in 32 bits except the two `181 *` products per pass (dct.ml:43-44,
// 87-88), which are formed in 64 bits.  That is exact whenever sum(|dequantised coefficient|) over the
// block is below HCJ_IDCT_L1_LIMIT (derivation in DESIGN.md; checked in tests/test_emul_idct.py).
// T = int64_t is the model's arithmetic verbatim and is taken for the (pathological) blocks above.
// ------------------------------------------------------------------------------------------------
#define HCJ_IDCT_L1_LIMIT HCJ_IDCT_L1_LIMIT_VALUE

template <typename T>
HCJ_HD T mul181(T a) {
  return (T)(((int64_t)a * 181 + 128) >> 8);
}

template <typename T, int STRIDE>
HCJ_HD void idct_row(T *b) {  // dct.ml:11-54
  const T W1 = 2841, W2 = 2676, W3 = 2408, W5 = 1609, W6 = 1108, W7 = 565;
  T x0 = b[0 * STRIDE] * 2048 + 128, x1 = b[4 * STRIDE] * 2048, x2 = b[6 * STRIDE], x3 = b[2 * STRIDE],
    x4 = b[1 * STRIDE], x5 = b[7 * STRIDE], x6 = b[5 * STRIDE], x7 = b[3 * STRIDE], x8;
  x8 = W7 * (x4 + x5);
  x4 = x8 + (W1 - W7) * x4;
  x5 = x8 - (W1 + W7) * x5;
  x8 = W3 * (x6 + x7);
  x6 = x8 - (W3 - W5) * x6;
  x7 = x8 - (W3 + W5) * x7;
  x8 = x0 + x1;
  x0 = x0 - x1;
  x1 = W6 * (x3 + x2);
  x2 = x1 - (W2 + W6) * x2;
  x3 = x1 + (W2 - W6) * x3;
  x1 = x4 + x6;
  x4 = x4 - x6;
  x6 = x5 + x7;
  x5 = x5 - x7;
  // third + fourth stage (dct.ml:39-53) written as three-input sums: x7 = x8 + x3, x8' = x8 - x3,
  // x3' = x0 + x2, x0' = x0 - x2 are only ever used inside the output sums, and two's-complement
  // addition is associative, so the results are bit-identical while an IADD3 does two adds at once.
  const T y2 = mul181<T>(x4 + x5);
  const T y4 = mul181<T>(x4 - x5);
  b[0 * STRIDE] = (x8 + x3 + x1) >> 8;
  b[1 * STRIDE] = (x0 + x2 + y2) >> 8;
  b[2 * STRIDE] = (x0 - x2 + y4) >> 8;
  b[3 * STRIDE] = (x8 - x3 + x6) >> 8;
  b[4 * STRIDE] = (x8 - x3 - x6) >> 8;
  b[5 * STRIDE] = (x0 - x2 - y4) >> 8;
  b[6 * STRIDE] = (x0 + x2 - y2) >> 8;
  b[7 * STRIDE] = (x8 + x3 - x1) >> 8;
}

// BIAS is added to every output before the final >> 14 (x0 reaches each output exactly once): with
// BIAS = 128 << 14 the outputs are the model's values + 128, i.e. the level shift of recon
// (decoder.ml:220) folded into the transform at no cost.
template <typename T, int STRIDE, int BIAS = 0>
HCJ_HD void idct_col(T *b) {  // dct.ml:56-98
  const T W1 = 2841, W2 = 2676, W3 = 2408, W5 = 1609, W6 = 1108, W7 = 565;
  T x0 = b[0 * STRIDE] * 256 + (8192 + BIAS), x1 = b[4 * STRIDE] * 256, x2 = b[6 * STRIDE], x3 = b[2 * STRIDE],
    x4 = b[1 * STRIDE], x5 = b[7 * STRIDE], x6 = b[5 * STRIDE], x7 = b[3 * STRIDE], x8;
  x8 = W7 * (x4 + x5) + 4;
  x4 = (x8 + (W1 - W7) * x4) >> 3;
  x5 = (x8 - (W1 + W7) * x5) >> 3;
  x8 = W3 * (x6 + x7) + 4;
  x6 = (x8 - (W3 - W5) * x6) >> 3;
  x7 = (x8 - (W3 + W5) * x7) >> 3;
  x8 = x0 + x1;
  x0 = x0 - x1;
  x1 = W6 * (x3 + x2) + 4;
  x2 = (x1 - (W2 + W6) * x2) >> 3;
  x3 = (x1 + (W2 - W6) * x3) >> 3;
  x1 = x4 + x6;
  x4 = x4 - x6;
  x6 = x5 + x7;
  x5 = x5 - x7;
  // third + fourth stage (dct.ml:83-97) written as three-input sums: x7 = x8 + x3, x8' = x8 - x3,
  // x3' = x0 + x2, x0' = x0 - x2 are only ever used inside the output sums, and two's-complement
  // addition is associative, so the results are bit-identical while an IADD3 does two adds at once.
  const T y2 = mul181<T>(x4 + x5);
  const T y4 = mul181<T>(x4 - x5);
  b[0 * STRIDE] = (x8 + x3 + x1) >> 14;
  b[1 * STRIDE] = (x0 + x2 + y2) >> 14;
  b[2 * STRIDE] = (x0 - x2 + y4) >> 14;
  b[3 * STRIDE] = (x8 - x3 + x6) >> 14;
  b[4 * STRIDE] = (x8 - x3 - x6) >> 14;
  b[5 * STRIDE] = (x0 - x2 - y4) >> 14;
  b[6 * STRIDE] = (x0 + x2 - y2) >> 14;
  b[7 * STRIDE] = (x8 + x3 - x1) >> 14;
}

template <typename T, int BIAS = 0>
HCJ_HD void idct_8x8(T v[64]) {  // dct.ml:100-107: all rows, then all columns
#pragma unroll
  for (int i = 0; i < 8; i++) idct_row<T, 1>(v + 8 * i);
#pragma unroll
  for (int i = 0; i < 8; i++) idct_col<T, 8, BIAS>(v + i);
}

// Four samples clamped to [0, 255] and packed little-endian (sample 0 in the low byte):
// clip to [-128, 127] then + 128 (decoder.ml:213-224) == clamp(v + 128, 0, 255).
HCJ_HD uint32_t pack4_sat(int32_t p0, int32_t p1, int32_t p2, int32_t p3) {
#if defined(__CUDA_ARCH__)
  uint32_t t, d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(p3), "r"(p2), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(p1), "r"(p0), "r"(t));
  return d;
#else
  auto c = [](int32_t v) { return (uint32_t)(v < 0 ? 0 : v > 255 ? 255 : v); };
  return c(p0) | (c(p1) << 8) | (c(p2) << 16) | (c(p3) << 24);
#endif
}

// Zigzag.inverse (zigzag.ml:3-69) as a compile-time function so that fully unrolled loops index
// registers, not memory.
HCJ_HD constexpr int zigzag_inverse(int i) {
  constexpr int t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                         41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                         30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
  return t[i];
}
// Zigzag.forward (zigzag.ml:71-137): natural index -> zig-zag position.
HCJ_HD constexpr int zigzag_forward(int i) {
  constexpr int t[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30,
                         41, 43, 9,  11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38,
                         46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};
  return t[i];
}

// dequantize + inverse zig-zag (decoder.ml:142-149), IDCT, clip and level shift (decoder.ml:213-224).
// cw[j]: zig-zag coefficients 2j (low half) and 2j+1 (high half) as int16, coefficient 0 the resolved DC;
// q[i]: quant table in file (zig-zag) order; out[2r], out[2r+1]: the 8 samples of row r, packed.
// The fast version works in 32 bits and returns false (leaving `out` unspecified) when the block's
// sum(|dequantised coefficient|) reaches HCJ_IDCT_L1_LIMIT; the caller then takes the wide version.
// lo16(cw) * q_lo and hi16(cw) * q_hi for quant entries <= 255: one dp2a each (signed halves of `cw`
// times the unsigned bytes 0 / 1 of the second operand), i.e. unpack + dequantise in one instruction.
// The table is kept in "dp2a form" (HCJ_QD): entry i holds q[i] for even i and q[i] << 8 for odd i.
#define HCJ_QD(i, q) (((i) & 1) ? (int32_t)(q) << 8 : (int32_t)(q))
HCJ_HD int32_t dequant_lo(uint32_t cw, int32_t q) {
#if defined(__CUDA_ARCH__)
  int32_t d;
  asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(cw), "r"(q), "r"(0));
  return d;
#else
  return (int32_t)(int16_t)(cw & 0xffffu) * q;
#endif
}
HCJ_HD int32_t dequant_hi(uint32_t cw, int32_t q) {
#if defined(__CUDA_ARCH__)
  int32_t d;
  asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(cw), "r"(q), "r"(0));
  return d;
#else
  return (int32_t)(int16_t)(cw >> 16) * (q >> 8);
#endif
}

// GUARD = false: the caller already knows the block is below the limit (wide-block flags written by
// the entropy decoders), so the sum is not formed.
template <bool GUARD = true>
HCJ_HD bool reconstruct_fast(const uint32_t cw[32], const int32_t *__restrict__ qd /* dp2a form */, uint32_t out[16]) {
  int32_t v[64];
  uint32_t l1 = 0;
#pragma unroll
  for (int j = 0; j < 32; j++) {
    int32_t d0 = dequant_lo(cw[j], qd[2 * j]), d1 = dequant_hi(cw[j], qd[2 * j + 1]);
    v[zigzag_inverse(2 * j)] = d0;
    v[zigzag_inverse(2 * j + 1)] = d1;
    if (GUARD) l1 += (uint32_t)(d0 < 0 ? -d0 : d0) + (uint32_t)(d1 < 0 ? -d1 : d1);
  }
  if (GUARD && l1 >= (uint32_t)HCJ_IDCT_L1_LIMIT) return false;
  idct_8x8<int32_t, (128 << 14)>(v);
#pragma unroll
  for (int r = 0; r < 8; r++) {
    out[2 * r] = pack4_sat(v[8 * r], v[8 * r + 1], v[8 * r + 2], v[8 * r + 3]);
    out[2 * r + 1] = pack4_sat(v[8 * r + 4], v[8 * r + 5], v[8 * r + 6], v[8 * r + 7]);
  }
  return true;
}

// The model's arithmetic verbatim (64-bit), for blocks above the guard or quant entries above 255.
HCJ_HD void reconstruct_wide(const uint32_t *cw, const int32_t *q, uint32_t *out) {
  int64_t w[64];
  for (int j = 0; j < 32; j++) {
    int64_t lo = (int16_t)(cw[j] & 0xffffu), hi = (int16_t)(cw[j] >> 16);
    w[zigzag_inverse(2 * j)] = lo * (int64_t)q[2 * j];
    w[zigzag_inverse(2 * j + 1)] = hi * (int64_t)q[2 * j + 1];
  }
  idct_8x8<int64_t>(w);
  for (int k = 0; k < 16; k++) {
    uint32_t word = 0;
    for (int i = 0; i < 4; i++) {
      int64_t sv = w[4 * k + i] < -128 ? -128 : w[4 * k + i] > 127 ? 127 : w[4 * k + i];
      word |= (uint32_t)(sv + 128) << (8 * i);
    }
    out[k] = word;
  }
}

// Convenience form used by the debug tap and the CPU emulation.
HCJ_HD void reconstruct_block(const int16_t c[64], const uint16_t q[64], bool force_wide, uint8_t pix[64]) {
  uint32_t cw[32], out[16];
  int32_t q32[64], qd[64];
  for (int j = 0; j < 32; j++) cw[j] = (uint32_t)(uint16_t)c[2 * j] | ((uint32_t)(uint16_t)c[2 * j + 1] << 16);
  for (int i = 0; i < 64; i++) {
    q32[i] = q[i];
    qd[i] = HCJ_QD(i, q[i]);
  }
  if (force_wide || !reconstruct_fast<true>(cw, qd, out)) reconstruct_wide(cw, q32, out);
  for (int k = 0; k < 64; k++) pix[k] = (uint8_t)(out[k >> 2] >> (8 * (k & 3)));
}

// ------------------------------------------------------------------------------------------------
// Scaled decode (HCJ_FLAG_SCALE_*): libjpeg's reduced inverse DCTs (jidctred.c jpeg_idct_4x4 / _2x2 / _1x1, CONST_BITS
// 13, PASS1_BITS 2), columns first, then rows, in exact integer arithmetic; out = clamp(x + 128, 0, 255).
// cw: the block as reconstruct_fast takes it; q: quant table in zig-zag order, plain values.  out[r]: the k samples of
// row r, packed little-endian.
// TC is the type of the column pass.  TC = int32_t is exact for blocks the entropy decoders did not flag (quant
// entries <= 255 and sum(|dequantised coefficient|) = L1 < HCJ_IDCT_L1_LIMIT): every column-pass value is a signed sum
// of dequantised coefficients of one column with weights of at most 20995 (4x4) / 32768 (2x2), so it stays below
// 32768 * 60000 + 4096 < 2^31.  The row pass always runs in 64 bits: its inputs can reach 5.2 L1 (4x4) / 4 L1 (2x2),
// which times its weights overflows 32 bits from L1 of about 20000 / 16000 on.  TC = int64_t (flagged blocks, 16-bit
// tables) is the reference arithmetic verbatim (DESIGN.md 4).
// ------------------------------------------------------------------------------------------------
template <typename T>
HCJ_HD T dequant_nat(const uint32_t cw[32], const int32_t *q, int n) {  // dequantised coefficient at natural index n
  const int z = zigzag_forward(n);
  const int32_t c = (z & 1) ? (int32_t)(int16_t)(cw[z >> 1] >> 16) : (int32_t)(int16_t)(cw[z >> 1] & 0xffffu);
  return (T)c * (T)q[z];
}

// One pass of jpeg_idct_4x4 over inputs 0, 1, 2, 3, 5, 6, 7 (input 4 does not contribute), descaled by `sh`.
template <typename T>
HCJ_HD void idct4_pass(T c0, T c1, T c2, T c3, T c5, T c6, T c7, int sh, T o[4]) {
  const T t0 = c0 * (T)(1 << 14);                          // << (CONST_BITS + 1)
  const T t2 = c2 * (T)15137 - c6 * (T)6270;               // FIX(1.847759065), FIX(0.765366865)
  const T t10 = t0 + t2, t12 = t0 - t2;
  const T a0 = c1 * (T)8697 - c3 * (T)17799 + c5 * (T)11893 - c7 * (T)1730;
  const T a2 = c1 * (T)20995 + c3 * (T)7373 - c5 * (T)4926 - c7 * (T)4176;
  const T r = (T)1 << (sh - 1);
  o[0] = (t10 + a2 + r) >> sh;
  o[1] = (t12 + a0 + r) >> sh;
  o[2] = (t12 - a0 + r) >> sh;
  o[3] = (t10 - a2 + r) >> sh;
}

// One pass of jpeg_idct_2x2 over inputs 0, 1, 3, 5, 7.
template <typename T>
HCJ_HD void idct2_pass(T c0, T c1, T c3, T c5, T c7, int sh, T o[2]) {
  const T t10 = c0 * (T)(1 << 15);                         // << (CONST_BITS + 2)
  const T t0 = c1 * (T)29692 - c3 * (T)10426 + c5 * (T)6967 - c7 * (T)5906;
  const T r = (T)1 << (sh - 1);
  o[0] = (t10 + t0 + r) >> sh;
  o[1] = (t10 - t0 + r) >> sh;
}

// A row-pass result + 128, clamped: with TC = int32_t it is below 2^15 in magnitude (see above), so the cast is exact.
template <typename TC>
HCJ_HD int32_t reduced_sample(int64_t v) {
  if (sizeof(TC) == 8) v = v < -128 ? -128 : v > 127 ? 127 : v;
  return (int32_t)v + 128;
}

template <typename TC>
HCJ_HD void reconstruct_4x4(const uint32_t cw[32], const int32_t *q, uint32_t out[4]) {
  int64_t ws[4][8];
#pragma unroll
  for (int c = 0; c < 8; c++) {
    if (c == 4) continue;  // column 4 is not read by the row pass
    TC o[4];
    idct4_pass<TC>(dequant_nat<TC>(cw, q, c), dequant_nat<TC>(cw, q, 8 + c), dequant_nat<TC>(cw, q, 16 + c),
                   dequant_nat<TC>(cw, q, 24 + c), dequant_nat<TC>(cw, q, 40 + c), dequant_nat<TC>(cw, q, 48 + c),
                   dequant_nat<TC>(cw, q, 56 + c), 12, o);  // CONST_BITS - PASS1_BITS + 1
#pragma unroll
    for (int r = 0; r < 4; r++) ws[r][c] = (int64_t)o[r];
  }
#pragma unroll
  for (int r = 0; r < 4; r++) {
    int64_t o[4];
    idct4_pass<int64_t>(ws[r][0], ws[r][1], ws[r][2], ws[r][3], ws[r][5], ws[r][6], ws[r][7], 19, o);  // CONST_BITS + PASS1_BITS + 3 + 1
    out[r] = pack4_sat(reduced_sample<TC>(o[0]), reduced_sample<TC>(o[1]), reduced_sample<TC>(o[2]), reduced_sample<TC>(o[3]));
  }
}

template <typename TC>
HCJ_HD void reconstruct_2x2(const uint32_t cw[32], const int32_t *q, uint32_t out[2]) {
  int64_t ws[2][8];
#pragma unroll
  for (int c = 1; c < 8; c += 2) {  // columns 1, 3, 5, 7 here, column 0 below; 2, 4, 6 are not read by the row pass
    TC o[2];
    idct2_pass<TC>(dequant_nat<TC>(cw, q, c), dequant_nat<TC>(cw, q, 8 + c), dequant_nat<TC>(cw, q, 24 + c),
                   dequant_nat<TC>(cw, q, 40 + c), dequant_nat<TC>(cw, q, 56 + c), 13, o);  // CONST_BITS - PASS1_BITS + 2
    ws[0][c] = (int64_t)o[0];
    ws[1][c] = (int64_t)o[1];
  }
  {
    TC o[2];
    idct2_pass<TC>(dequant_nat<TC>(cw, q, 0), dequant_nat<TC>(cw, q, 8), dequant_nat<TC>(cw, q, 24), dequant_nat<TC>(cw, q, 40),
                   dequant_nat<TC>(cw, q, 56), 13, o);
    ws[0][0] = (int64_t)o[0];
    ws[1][0] = (int64_t)o[1];
  }
#pragma unroll
  for (int r = 0; r < 2; r++) {
    int64_t o[2];
    idct2_pass<int64_t>(ws[r][0], ws[r][1], ws[r][3], ws[r][5], ws[r][7], 20, o);  // CONST_BITS + PASS1_BITS + 3 + 2
    out[r] = pack4_sat(reduced_sample<TC>(o[0]), reduced_sample<TC>(o[1]), 0, 0);
  }
}

// jpeg_idct_1x1: DESCALE(dc * q, 3).  Exact in 32 bits for any int16 DC and 16-bit quant entry (|dc q| + 4 < 2^31).
HCJ_HD uint32_t reconstruct_1x1(uint32_t cw0, int32_t q0) {
  const int32_t d = (int32_t)(int16_t)(cw0 & 0xffffu) * q0;
  return pack4_sat(((d + 4) >> 3) + 128, 0, 0, 0);
}

// The whole scaled reconstruction of one block as the IDCT kernel selects it (wide: the block is flagged or the image
// has quant entries above 255).  k = 4, 2, 1; out[r] as above.
HCJ_HD void reconstruct_scaled(const uint32_t cw[32], const int32_t *q, int k, bool wide, uint32_t *out) {
  if (k == 1) out[0] = reconstruct_1x1(cw[0], q[0]);
  else if (k == 2) wide ? reconstruct_2x2<int64_t>(cw, q, out) : reconstruct_2x2<int32_t>(cw, q, out);
  else wide ? reconstruct_4x4<int64_t>(cw, q, out) : reconstruct_4x4<int32_t>(cw, q, out);
}

// ------------------------------------------------------------------------------------------------
// libjpeg reconstruction (HCJ_FLAG_LIBJPEG): jidctint.c jpeg_idct_islow (CONST_BITS 13, PASS1_BITS 2), columns first,
// on the dequantised coefficients.  The column pass's results are stored as C int (truncated to 32 bits); the row
// pass's, descaled by 18, index libjpeg's range-limit table: sample = clamp(((v + 512) & 1023) - 512 + 128, 0, 255).
// That depends on bits 0..27 of the row pass's sum only, so the row pass is exact in wrapping 32-bit arithmetic for
// every block.  The column pass is exact in wrapping 32-bit arithmetic when its sums fit 32 bits: for blocks the
// entropy decoders did not flag (quant entries <= 255, sum(|dequantised coefficient|) = L1 < HCJ_IDCT_L1_LIMIT) they
// are at most 11363 L1 + 1024 < 2^30 (DESIGN.md 4).  Flagged blocks and 16-bit tables take the column pass in 64 bits
// (islow_wide).  T = uint32_t is the wrapping arithmetic, T = int64_t the C code's JLONG.
// ------------------------------------------------------------------------------------------------
// One islow pass over inputs c0..c7 (the even part, then the odd part of jidctint.c), before the descale.
template <typename T>
HCJ_HD void islow_pass(T c0, T c1, T c2, T c3, T c4, T c5, T c6, T c7, T o[8]) {
  const T z1 = (c2 + c6) * (T)4433;                                  // FIX_0_541196100
  const T t2 = z1 + c6 * (T)-15137, t3 = z1 + c2 * (T)6270;          // FIX_1_847759065, FIX_0_765366865
  const T t0 = (c0 + c4) * (T)8192, t1 = (c0 - c4) * (T)8192;       // << CONST_BITS
  const T t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  const T z5 = (c7 + c3 + c5 + c1) * (T)9633;                        // FIX_1_175875602
  const T za = (c7 + c1) * (T)-7373, zb = (c5 + c3) * (T)-20995;     // FIX_0_899976223, FIX_2_562915447
  const T zc = (c7 + c3) * (T)-16069 + z5, zd = (c5 + c1) * (T)-3196 + z5;  // FIX_1_961570560, FIX_0_390180644
  const T p0 = c7 * (T)2446 + za + zc, p1 = c5 * (T)16819 + zb + zd;  // FIX_0_298631336, FIX_2_053119869
  const T p2 = c3 * (T)25172 + zb + zc, p3 = c1 * (T)12299 + za + zd; // FIX_3_072711738, FIX_1_501321110
  o[0] = t10 + p3, o[7] = t10 - p3, o[1] = t11 + p2, o[6] = t11 - p2;
  o[2] = t12 + p1, o[5] = t12 - p1, o[3] = t13 + p0, o[4] = t13 - p0;
}

// DESCALE(x, CONST_BITS - PASS1_BITS) stored as C int.
HCJ_HD int32_t islow_ws(uint32_t v) { return (int32_t)(v + 1024u) >> 11; }
HCJ_HD int32_t islow_ws(int64_t v) { return (int32_t)((v + 1024) >> 11); }
// range_limit[DESCALE(x, CONST_BITS + PASS1_BITS + 3) & RANGE_MASK] before the final clamp (pack4_sat): adding 2^27
// moves the wrap point of the 10-bit index from 0 to -512.
HCJ_HD int32_t islow_sample(uint32_t v) { return (int32_t)(((v + (1u << 17) + (1u << 27)) >> 18) & 1023u) - 384; }

// Row pass of the islow block ws[64] (natural order, C int), packed into out[2r], out[2r + 1] as reconstruct_fast.
HCJ_HD void islow_rows(const int32_t ws[64], uint32_t out[16]) {
#pragma unroll
  for (int r = 0; r < 8; r++) {
    const int32_t *w = ws + 8 * r;
    uint32_t o[8];
    islow_pass<uint32_t>(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o);
    out[2 * r] = pack4_sat(islow_sample(o[0]), islow_sample(o[1]), islow_sample(o[2]), islow_sample(o[3]));
    out[2 * r + 1] = pack4_sat(islow_sample(o[4]), islow_sample(o[5]), islow_sample(o[6]), islow_sample(o[7]));
  }
}

// Unflagged blocks, quant entries <= 255: the table in dp2a form (HCJ_QD), as reconstruct_fast takes it.
HCJ_HD void islow_fast(const uint32_t cw[32], const int32_t *__restrict__ qd, uint32_t out[16]) {
  int32_t v[64];
#pragma unroll
  for (int j = 0; j < 32; j++) {
    v[zigzag_inverse(2 * j)] = dequant_lo(cw[j], qd[2 * j]);
    v[zigzag_inverse(2 * j + 1)] = dequant_hi(cw[j], qd[2 * j + 1]);
  }
#pragma unroll
  for (int c = 0; c < 8; c++) {
    uint32_t o[8];
    islow_pass<uint32_t>(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c], o);
#pragma unroll
    for (int r = 0; r < 8; r++) v[8 * r + c] = islow_ws(o[r]);
  }
  islow_rows(v, out);
}

// Any block, any 16-bit table: q plain, zig-zag order.  The column pass is jidctint.c's JLONG arithmetic verbatim.
HCJ_HD void islow_wide(const uint32_t *cw, const int32_t *q, uint32_t *out) {
  int32_t ws[64];
  for (int c = 0; c < 8; c++) {
    int64_t o[8];
    islow_pass<int64_t>(dequant_nat<int64_t>(cw, q, c), dequant_nat<int64_t>(cw, q, 8 + c), dequant_nat<int64_t>(cw, q, 16 + c),
                        dequant_nat<int64_t>(cw, q, 24 + c), dequant_nat<int64_t>(cw, q, 32 + c), dequant_nat<int64_t>(cw, q, 40 + c),
                        dequant_nat<int64_t>(cw, q, 48 + c), dequant_nat<int64_t>(cw, q, 56 + c), o);
    for (int r = 0; r < 8; r++) ws[8 * r + c] = islow_ws(o[r]);
  }
  islow_rows(ws, out);
}

// libjpeg's up-sampling (jdsample.c, do_fancy_upsampling) of one component to output sample (x, y).  p: the component's
// plane (pitch bytes per row) of which rw x rh samples are real (ceil(W / hr) x ceil(H / vr)); (hr, vr) = (h_max / h_c,
// v_max / v_c).  The fancy filters clamp their neighbours to the real plane, which gives libjpeg's edge columns and
// its replicated context rows.  h2v1 / h2v2 replicate instead when the real plane is at most 2 samples wide.
HCJ_HD int libjpeg_upsample(const uint8_t *p, int pitch, int rw, int rh, int hr, int vr, int x, int y) {
  const int j = x / hr, i = y / vr;
  int jn = j + ((x & 1) ? 1 : -1), ni = i + ((y & 1) ? 1 : -1);
  jn = jn < 0 ? 0 : jn > rw - 1 ? rw - 1 : jn;
  ni = ni < 0 ? 0 : ni > rh - 1 ? rh - 1 : ni;
  const int a = p[(int64_t)i * pitch + j];
  if (hr == 1 && vr == 2) return (3 * a + p[(int64_t)ni * pitch + j] + 1 + (y & 1)) >> 2;           // h1v2_fancy_upsample
  if (hr == 2 && vr == 1 && rw > 2) return (3 * a + p[(int64_t)i * pitch + jn] + 1 + (x & 1)) >> 2;  // h2v1_fancy_upsample
  if (hr == 2 && vr == 2 && rw > 2) {                                                             // h2v2_fancy_upsample
    const int cs = 3 * a + p[(int64_t)ni * pitch + j], cn = 3 * p[(int64_t)i * pitch + jn] + p[(int64_t)ni * pitch + jn];
    return (3 * cs + cn + 8 - (x & 1)) >> 4;
  }
  return a;  // fullsize_upsample, h2v1 / h2v2_upsample, int_upsample
}

// ------------------------------------------------------------------------------------------------
// Dct.Chen.forward_8x8 (dct.ml:109-196): columns first, then rows.  Inputs are pixel - 128, so 32-bit
// arithmetic is exact (|value| < 2^21 throughout).
// ------------------------------------------------------------------------------------------------
HCJ_HD int32_t fc4(int32_t f, int32_t g) { return (362 * (f + g)) >> 9; }
HCJ_HD int32_t fc62(int32_t f, int32_t g) { return (196 * f + 473 * g) >> 9; }
HCJ_HD int32_t fc71(int32_t f, int32_t g) { return (100 * f + 502 * g) >> 9; }
HCJ_HD int32_t fc35(int32_t f, int32_t g) { return (426 * f + 284 * g) >> 9; }

template <int STRIDE>
HCJ_HD void fdct_1d(int32_t *b) {  // dct.ml:114-149 / :151-187
  int32_t a0 = b[0 * STRIDE] + b[7 * STRIDE], c3 = b[0 * STRIDE] - b[7 * STRIDE];
  int32_t a1 = b[1 * STRIDE] + b[6 * STRIDE], c2 = b[1 * STRIDE] - b[6 * STRIDE];
  int32_t a2 = b[2 * STRIDE] + b[5 * STRIDE], c1 = b[2 * STRIDE] - b[5 * STRIDE];
  int32_t a3 = b[3 * STRIDE] + b[4 * STRIDE], c0 = b[3 * STRIDE] - b[4 * STRIDE];
  int32_t b0 = a0 + a3, b1 = a1 + a2, b2 = a1 - a2, b3 = a0 - a3;
  b[0 * STRIDE] = fc4(b0, b1);
  b[4 * STRIDE] = fc4(b0, -b1);
  b[2 * STRIDE] = fc62(b2, b3);
  b[6 * STRIDE] = fc62(b3, -b2);
  b0 = fc4(c2, -c1);
  b1 = fc4(c2, c1);
  a0 = c0 + b0;
  a1 = c0 - b0;
  a2 = c3 - b1;
  a3 = c3 + b1;
  b[1 * STRIDE] = fc71(a0, a3);
  b[5 * STRIDE] = fc35(a1, a2);
  b[3 * STRIDE] = fc35(a2, -a1);
  b[7 * STRIDE] = fc71(a3, -a0);
}

HCJ_HD void fdct_8x8(int32_t v[64]) {
#pragma unroll
  for (int i = 0; i < 8; i++) fdct_1d<8>(v + i);
#pragma unroll
  for (int i = 0; i < 8; i++) fdct_1d<1>(v + 8 * i);
}

// Encoder.quant_and_scale (encoder.ml:98-101): (f -/+ 2q) / (4q), OCaml's truncating division,
// computed with a reciprocal: recip = floor(2^32 / (4q)) + 1 is exact for |f| + 2q < 2^20
// (checked exhaustively in tests/test_emul_encode.py).
HCJ_HD int32_t quantize(int32_t f, uint32_t q, uint32_t recip) {
  uint32_t n = (uint32_t)(f < 0 ? -f : f) + 2u * q;
#if defined(__CUDA_ARCH__)
  uint32_t d = __umulhi(n, recip);
#else
  uint32_t d = (uint32_t)(((uint64_t)n * recip) >> 32);
#endif
  return f < 0 ? -(int32_t)d : (int32_t)d;
}

// Encoder.size (encoder.ml:143) and Encoder.magnitude (encoder.ml:145-147).
HCJ_HD uint32_t coef_size(int32_t v) {
  uint32_t a = (uint32_t)(v < 0 ? -v : v);
#if defined(__CUDA_ARCH__)
  return 32u - (uint32_t)__clz((int)a);
#else
  uint32_t s = 0;
  while (a) {
    s++;
    a >>= 1;
  }
  return s;
#endif
}
HCJ_HD uint32_t coef_magnitude(int32_t v, uint32_t size) {
  return (uint32_t)(v >= 0 ? v : v - 1) & ((1u << size) - 1u);
}

}  // namespace hcjdev

namespace hcjdev {

// ------------------------------------------------------------------------------------------------
// Encoder.rle + write_bits (encoder.ml:127-193) for one block: calls emit(bits, nbits) for every
// field the model passes to Writer.put_bits, in order.  q: quantised zig-zag block (q[0] ignored),
// dcdiff: quant.(0) - dc_pred.  dc_codes[size], ac_codes[(run << 4) | size] = (code << 8) | length.
// Returns false if a symbol has no code (the model raises an index-out-of-bounds exception).
// ------------------------------------------------------------------------------------------------
// `coef(k)` returns quantised coefficient k (zig-zag order).  The loop over k is written to be fully unrolled, so
// that a kernel can keep the block in registers (coef(k) with a constant k) instead of a local-memory array.
// WITH_DC = false emits the AC fields only (the DC differential needs the neighbouring block's DC).
template <bool WITH_DC = true, class Coef, class Emit>
HCJ_HD bool encode_block_fields_from(Coef coef, int32_t dcdiff, const uint32_t *dc_codes, const uint32_t *ac_codes, Emit &emit) {
  bool ok = true;
  uint32_t size, code;
  if (WITH_DC) {
    size = coef_size(dcdiff);
    code = size < 16u ? dc_codes[size] : 0u;
    ok &= (code & 0xffu) != 0u;
    emit(code >> 8, code & 0xffu);
    emit(coef_magnitude(dcdiff, size), size);
  }
  uint32_t run = 0;
#pragma unroll
  for (int k = 1; k < 64; k++) {
    const int32_t v = coef(k);
    if (k == 63 && v == 0) {  // [ { run; value = 0 } ] -> end of block (encoder.ml:172-175)
      code = ac_codes[0x00];
      ok &= (code & 0xffu) != 0u;
      emit(code >> 8, code & 0xffu);
    } else if (v != 0) {
      for (; run >= 16u; run -= 16u) {  // runs (encoder.ml:178-185)
        code = ac_codes[0xf0];
        ok &= (code & 0xffu) != 0u;
        emit(code >> 8, code & 0xffu);
      }
      size = coef_size(v);
      code = size < 16u ? ac_codes[(run << 4) | size] : 0u;
      ok &= (code & 0xffu) != 0u;
      emit(code >> 8, code & 0xffu);
      emit(coef_magnitude(v, size), size);
      run = 0;
    } else {
      run++;
    }
  }
  return ok;
}

template <class Emit>
HCJ_HD bool encode_block_fields(const int16_t *q, int32_t dcdiff, const uint32_t *dc_codes, const uint32_t *ac_codes,
                                Emit &emit) {
  return encode_block_fields_from([q](int k) { return (int32_t)q[k]; }, dcdiff, dc_codes, ac_codes, emit);
}

// ------------------------------------------------------------------------------------------------
// The same field sequence driven by the block's non-zero map: one iteration per non-zero AC coefficient
// instead of 63 (a 1080p q75 block has about ten).  Fully unrolled over k the loop above is ~2500
// instructions of branchy code per block, which the encoder kernels could not fetch fast enough (ncu:
// 7.4 "no instruction" stall cycles per issue in k_pack, 14 of 32 lanes active); this one is a short loop.
// `nz`: bit k set iff coefficient k != 0; `coef(k)`: the value, k chosen at run time.
// ------------------------------------------------------------------------------------------------
HCJ_HD uint64_t nonzero_map(const uint32_t qw[32]) {  // qw[j] = coefficients 2j (low half) and 2j + 1
  uint64_t m = 0;
#pragma unroll
  for (int g = 0; g < 8; g++) {
    uint32_t a = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const uint32_t w = qw[4 * g + i];
      a |= (((w & 0xffffu) ? 1u : 0u) | ((w >> 16) ? 2u : 0u)) << (2 * i);
    }
    m |= (uint64_t)a << (8 * g);
  }
  return m;
}
HCJ_HD int lowest_bit(uint64_t m) {
#if defined(__CUDA_ARCH__)
  return __ffsll((long long)m) - 1;
#else
  return __builtin_ctzll(m);
#endif
}
// A code and the magnitude bits behind it leave as ONE field (at most 16 + 15 bits): half the calls into the packer.
template <class Coef, class Emit>
HCJ_HD bool encode_block_fields_sparse(uint64_t nz, Coef coef, int32_t dcdiff, const uint32_t *dc_codes, const uint32_t *ac_codes,
                                       Emit &emit) {
  bool ok = true;
  uint32_t size = coef_size(dcdiff);
  uint32_t code = size < 16u ? dc_codes[size] : 0u;
  ok &= (code & 0xffu) != 0u;
  emit(((code >> 8) << size) | coef_magnitude(dcdiff, size), (code & 0xffu) + size);
  int prev = 0;  // position of the previous non-zero coefficient (the DC slot to start with)
  for (uint64_t m = nz & ~1ull; m; m &= m - 1ull) {
    const int k = lowest_bit(m);
    uint32_t run = (uint32_t)(k - prev - 1);
    prev = k;
    const int32_t v = coef(k);
    for (; run >= 16u; run -= 16u) {  // runs (encoder.ml:178-185)
      code = ac_codes[0xf0];
      ok &= (code & 0xffu) != 0u;
      emit(code >> 8, code & 0xffu);
    }
    size = coef_size(v);
    code = size < 16u ? ac_codes[(run << 4) | size] : 0u;
    ok &= (code & 0xffu) != 0u;
    emit(((code >> 8) << size) | coef_magnitude(v, size), (code & 0xffu) + size);
  }
  if (prev != 63) {  // coefficient 63 is zero: [ { run; value = 0 } ] -> end of block (encoder.ml:172-175)
    code = ac_codes[0x00];
    ok &= (code & 0xffu) != 0u;
    emit(code >> 8, code & 0xffu);
  }
  return ok;
}

// coefficient k of a block held as 32 words of two int16 each (the layout of the coefficient buffer)
HCJ_HD int32_t packed_coef(const uint32_t *qw, int k) {
  const uint32_t w = qw[k >> 1];
  return (k & 1) ? (int32_t)w >> 16 : (int32_t)(int16_t)(w & 0xffffu);
}


// ------------------------------------------------------------------------------------------------
// Stated forward colour conversion (DESIGN.md 5; not in the reference): JFIF full range, libjpeg's jccolor.c in 16-bit
// fixed point.  Returns the sums before the shift: sample = t >> 16, and every t lies in [0, 2^24), so the sample is
// byte 2 of t and no clamp is needed (all 2^24 triples checked, tests/test_encode_rgb.py).
// ------------------------------------------------------------------------------------------------
HCJ_HD void rgb_to_ycc_fixed(int r, int g, int b, int &ty, int &tcb, int &tcr) {
  ty = 19595 * r + 38470 * g + 7471 * b + 32768;
  tcb = -11059 * r - 21709 * g + 32768 * b + ((128 << 16) + 32767);
  tcr = 32768 * r - 27439 * g - 5329 * b + ((128 << 16) + 32767);
}

#if defined(__CUDACC__)
// NW words to `nbytes` bytes at any address: 16-byte stores when the address allows and all bytes are wanted,
// 4-byte stores when it is word aligned, bytes otherwise (and for the tail).
template <int NW>
__device__ __forceinline__ void store_any(uint8_t *dst, const uint32_t (&w)[NW], int nbytes) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(dst);
  if (NW % 4 == 0 && (a & 15u) == 0 && nbytes == NW * 4) {
#pragma unroll
    for (int k = 0; k < NW / 4; k++) reinterpret_cast<uint4 *>(dst)[k] = make_uint4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
  } else if ((a & 3u) == 0) {
#pragma unroll
    for (int k = 0; k < NW; k++) {
      if (4 * k + 4 <= nbytes) {
        reinterpret_cast<uint32_t *>(dst)[k] = w[k];
      } else {
#pragma unroll
        for (int i = 0; i < 4; i++)
          if (4 * k + i < nbytes) dst[4 * k + i] = (uint8_t)(w[k] >> (8 * i));
      }
    }
  } else {
    // not word aligned: up to three head bytes, then the words of the byte sequence shifted by the head (funnel
    // shifts over neighbouring words), then up to three tail bytes - instead of a byte store per byte
    const int head = (4 - (int)(a & 3u)) & 3, sh = 8 * head;
#pragma unroll
    for (int i = 0; i < 3; i++)
      if (i < head && i < nbytes) dst[i] = (uint8_t)(w[0] >> (8 * i));
    const int nw = nbytes > head ? (nbytes - head) >> 2 : 0;
    uint32_t *d32 = reinterpret_cast<uint32_t *>(dst + head);
    uint32_t tail = 0;
#pragma unroll
    for (int k = 0; k < NW; k++) {
      const uint32_t v = __funnelshift_r(w[k], k + 1 < NW ? w[k + 1] : 0u, sh);  // bytes head + 4k .. head + 4k + 3
      if (k < nw) d32[k] = v;
      if (k == nw) tail = v;
    }
    const int done = head + 4 * nw;
#pragma unroll
    for (int i = 0; i < 3; i++)
      if (done + i < nbytes) dst[done + i] = (uint8_t)(tail >> (8 * i));
  }
}
#endif

}  // namespace hcjdev
