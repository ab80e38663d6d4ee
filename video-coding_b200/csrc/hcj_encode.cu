// hcj_encode.cu — encoder mirror (Encoder.encode_420/422/444, jpeg/model/src/encoder.ml) for sm_100a.
//
//   k_fdct_quant   E2,E4-E6  zero-padded block fetch, level shift, Chen FDCT, quantise, zig-zag
//   k_block_bits   E7,E8     per block: DC differential + (run, size) symbols -> the block's code + magnitude fields packed
//                            into its own 512-bit slot, and their length in bits (the field loop runs once per block:
//                            the block staged in shared memory, one iteration per non-zero coefficient,
//                            encode_block_fields_sparse)
//   k_symbol_counts  HCJ_ENC_OPTIMIZE_HUFFMAN only, before k_block_bits: per frame and table, the counts of the symbols the
//                    default encode codes (block_symbols_sparse)
//   k_huff_tables    HCJ_ENC_OPTIMIZE_HUFFMAN only: per frame, libjpeg's K.2 tables (one warp per table) as the codes
//                    k_block_bits / k_pack read, and the frame's header with those DHT segments, which k_seg_scan copies
//   k_scan_bits    per frame: exclusive prefix sum of block bit lengths (one CTA walks the frame)
//   k_place        E8,E9     per block: the finished bit string shifted to its bit offset (big-endian 32-bit words,
//                            atomicOr only on the two boundary words), 1-fill at the end of every segment
//                            (flush_with_1s, bitstream_writer.ml:45-49)
//   k_pack         E8,E9     blocks longer than their slot: the field loop again, straight to the bit offset (only
//                            launched when a chunk holds such a block)
//   k_seg_count    E9        per unit (segment, or 1 KiB of a lone segment): stuffed byte count
//   k_seg_scan     per frame: prefix sum of unit sizes -> output offsets; copies the header
//   k_stuff        E9,E10    per unit: byte copy with FF -> FF 00, RSTn between segments, EOI
//   k_rgb_to_ycc   K10       RGB24 input only (hcj_encode_rgb_batch): stated RGB -> YCbCr + Planar_444.convert_to_420 / _422
//                            into the planar frame buffer k_fdct_quant reads, from uploaded frames or the caller's device buffers
//
// Results are byte-identical to the model's Writer.get_buffer (tests/test_gpu_encode.py).
#include <cuda_runtime.h>
#include <string.h>

#include <new>
#include <thread>
#include <vector>

#include "hcj_device.cuh"
#include "hcj_host.h"
#include "hcj_internal.h"
#include "hcj_kernels.cuh"

namespace hcjk {
using namespace hcjdev;

// Rows of 144 bytes per thread / block in shared memory: 16-byte aligned, and conflict free for per-thread 16-byte accesses.
constexpr int ENC_ROW_WORDS = 36;

// ---- K6 ------------------------------------------------------------------------------------------
// One thread per block.  The quant table and its reciprocals come from shared memory (16-byte reads: they were 128
// scalar loads per block through L1), and the finished blocks leave through shared memory as one contiguous 16 KiB
// run per CTA (a thread storing its own 128-byte block costs eight L1 wavefronts per store instruction; the LSU data
// pipe was 82 % busy).
__global__ void __launch_bounds__(128) k_fdct_quant(EncodeBatchDev e) {
  __shared__ __align__(16) uint32_t s_rows[128 * ENC_ROW_WORDS];
  __shared__ __align__(16) uint16_t s_qt[2][64];
  __shared__ __align__(16) uint32_t s_qr[2][64];
  s_qt[threadIdx.x >> 6][threadIdx.x & 63] = e.qt[threadIdx.x];
  s_qr[threadIdx.x >> 6][threadIdx.x & 63] = e.qrecip[threadIdx.x];
  __syncthreads();
  const uint32_t blk0 = blockIdx.x * blockDim.x, blk = blk0 + threadIdx.x;
  const uint32_t frame = blockIdx.y;
  if (blk < e.nblocks) {
    const uint32_t mcu = blk / e.bpm, k = blk - mcu * e.bpm;
    const int c = e.blk_comp[k];
    const int my = mcu / e.mcus_wide, mx = mcu - my * e.mcus_wide;
    const int x0 = (mx * e.hs[c] + e.blk_bx[k]) * 8, y0 = (my * e.vs[c] + e.blk_by[k]) * 8;
    const uint8_t *src = e.src + (uint64_t)frame * e.frame_bytes + e.src_off[c];
    const int sw = e.src_w[c], sh = e.src_h[c];
    int32_t v[64];
    // level_shifted_input_block over the zero-initialised padded plane (encoder.ml:81-90, plane.ml:11-17)
    const bool inside = x0 + 8 <= sw && y0 + 8 <= sh;
    if (e.linear_blit && sw != e.plane_w[c]) {
      // encode_monochrome fills its padded plane with Plane.blit: ONE linear copy of the source bytes (encoder.ml:548,
      // plane.ml:20), so with a width that is not a multiple of 8 the rows of the plane are not the rows of the frame
      const int pw = e.plane_w[c];
      const int64_t nsrc = (int64_t)sw * sh;
#pragma unroll
      for (int y = 0; y < 8; y++)
#pragma unroll
        for (int x = 0; x < 8; x++) {
          const int64_t at = (int64_t)(y0 + y) * pw + (x0 + x);
          v[y * 8 + x] = (at < nsrc ? (int)__ldg(src + at) : 0) - 128;
        }
    } else if (inside && ((((uintptr_t)src + (size_t)y0 * sw + x0) & 7u) == 0) && (sw & 7) == 0) {
#pragma unroll
      for (int y = 0; y < 8; y++) {
        uint2 u = __ldg(reinterpret_cast<const uint2 *>(src + (size_t)(y0 + y) * sw + x0));
#pragma unroll
        for (int x = 0; x < 4; x++) {
          v[y * 8 + x] = (int32_t)((u.x >> (8 * x)) & 0xffu) - 128;
          v[y * 8 + 4 + x] = (int32_t)((u.y >> (8 * x)) & 0xffu) - 128;
        }
      }
    } else {
#pragma unroll
      for (int y = 0; y < 8; y++)
#pragma unroll
        for (int x = 0; x < 8; x++) {
          int px = x0 + x, py = y0 + y;
          int p = (px < sw && py < sh) ? (int)__ldg(src + (size_t)py * sw + px) : 0;
          v[y * 8 + x] = p - 128;
        }
    }
    fdct_8x8(v);
    const uint4 *qt4 = reinterpret_cast<const uint4 *>(s_qt[c ? 1 : 0]);
    const uint4 *qr4 = reinterpret_cast<const uint4 *>(s_qr[c ? 1 : 0]);
    uint4 *row = reinterpret_cast<uint4 *>(s_rows + threadIdx.x * ENC_ROW_WORDS);
#pragma unroll
    for (int g = 0; g < 8; g++) {  // quant (encoder.ml:103-108): zig-zag position z <- natural inverse(z), eight at a time
      const uint4 q = qt4[g], ra = qr4[2 * g], rb = qr4[2 * g + 1];
      const uint32_t qq[8] = {q.x & 0xffffu, q.x >> 16, q.y & 0xffffu, q.y >> 16, q.z & 0xffffu, q.z >> 16, q.w & 0xffffu, q.w >> 16};
      const uint32_t rr[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
      uint32_t o[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int z = 8 * g + 2 * i;
        const int32_t a = quantize(v[zigzag_inverse(z)], qq[2 * i], rr[2 * i]);
        const int32_t b = quantize(v[zigzag_inverse(z + 1)], qq[2 * i + 1], rr[2 * i + 1]);
        o[i] = ((uint32_t)a & 0xffffu) | ((uint32_t)b << 16);
      }
      row[g] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
  __syncthreads();
  uint4 *dst = reinterpret_cast<uint4 *>(e.quant + ((uint64_t)frame * e.nblocks + blk0) * 64);
  const uint32_t nchunks = min(128u, e.nblocks - blk0) * 8u;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t c = threadIdx.x + 128u * i;
    if (c < nchunks) dst[c] = *reinterpret_cast<const uint4 *>(s_rows + (c >> 3) * ENC_ROW_WORDS + (c & 7u) * 4u);
  }
}

// Index (within the frame) of the block whose DC is this block's predictor, or -1 (start of a segment).
__device__ __forceinline__ int64_t dc_pred_block(const EncodeBatchDev &e, uint32_t blk) {
  const uint32_t mcu = blk / e.bpm, k = blk - mcu * e.bpm;
  const int c = e.blk_comp[k];
  if (e.blk_bx[k] != 0 || e.blk_by[k] != 0) return (int64_t)blk - 1;  // previous block of the same component, same MCU
  if (mcu == 0 || (e.restart_interval && mcu % e.restart_interval == 0)) return -1;
  // last block of component c in the previous MCU
  uint32_t first = 0;
  for (int j = 0; j < c; j++) first += e.hs[j] * e.vs[j];
  return (int64_t)(mcu - 1) * e.bpm + first + e.hs[c] * e.vs[c] - 1;
}

struct BitCounter {
  uint32_t bits = 0;
  __device__ __forceinline__ void operator()(uint32_t, uint32_t n) { bits += n; }
};

struct EncTablesSmem {
  uint32_t dc[2][16];
  uint32_t ac[2][256];
};

__device__ __forceinline__ void load_enc_tables(EncTablesSmem &t, const EncodeBatchDev &e, uint32_t frame) {
  const uint32_t *dc = e.dc_codes + (uint64_t)frame * e.tab_stride, *ac = e.ac_codes + (uint64_t)frame * e.tab_stride;
  for (int i = threadIdx.x; i < 32; i += blockDim.x) t.dc[i >> 4][i & 15] = dc[i];
  for (int i = threadIdx.x; i < 512; i += blockDim.x) t.ac[i >> 8][i & 255] = ac[i];
}

// The 128 blocks of a CTA are one contiguous 16 KiB run of the coefficient buffer: the CTA copies it into shared memory
// with fully coalesced 16-byte loads (a thread reading its own 128-byte block costs eight L1 wavefronts per load
// instruction, and the LSU data pipe was what bound these kernels: 80 % busy), into rows of 144 bytes (16-byte
// aligned, conflict free for the per-thread 16-byte reads).  Each thread then takes its row: the non-zero map from
// eight 16-byte reads, single coefficients by a run-time index in the field loop.  Ends with a CTA barrier.
__device__ __forceinline__ void stage_cta_blocks(const int16_t *frame_quant, uint32_t blk0, uint32_t nblocks, uint32_t *s_rows) {
  const uint4 *src = reinterpret_cast<const uint4 *>(frame_quant + (uint64_t)blk0 * 64);
  const uint32_t nchunks = min(128u, nblocks - blk0) * 8u;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const uint32_t c = threadIdx.x + 128u * i;
    if (c < nchunks) *reinterpret_cast<uint4 *>(s_rows + (c >> 3) * ENC_ROW_WORDS + (c & 7u) * 4u) = __ldg(src + c);
  }
  __syncthreads();
}
__device__ __forceinline__ uint64_t row_nonzero_map(const uint32_t *row) {
  uint32_t qw[32];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const uint4 u = reinterpret_cast<const uint4 *>(row)[j];
    qw[4 * j] = u.x, qw[4 * j + 1] = u.y, qw[4 * j + 2] = u.z, qw[4 * j + 3] = u.w;
  }
  return nonzero_map(qw);
}

// The block's fields packed into its own slot, first bit in bit 31 of word 0: the field loop runs ONCE per block (it used to
// run in k_block_bits for the length and again in k_pack for the bits: 1.25 + 1.71 ms per 512 x 1080p); k_place only
// shifts the finished string to the block's bit offset.  Blocks longer than the slot keep the two-loop path (k_pack).
struct LocalPacker {
  uint32_t *slot;
  uint64_t acc;   // pending bits, right-aligned
  uint32_t nacc;  // number of pending bits (< 32 between calls)
  uint32_t widx;  // next word of the slot
  uint32_t bits;  // length so far
  __device__ __forceinline__ void init(uint32_t *slot_) {
    slot = slot_;
    acc = 0;
    nacc = widx = bits = 0;
  }
  __device__ __forceinline__ void operator()(uint32_t field, uint32_t n) {
    if (n == 0) return;
    acc = (acc << n) | (uint64_t)(field & ((1u << n) - 1u));
    nacc += n;
    bits += n;
    if (nacc >= 32u) {
      nacc -= 32u;
      if (widx < (uint32_t)HCJ_ENC_SLOT_WORDS) slot[widx] = (uint32_t)(acc >> nacc);
      widx++;
      acc &= (1ull << nacc) - 1ull;
    }
  }
  __device__ __forceinline__ void finish() {
    if (nacc && widx < (uint32_t)HCJ_ENC_SLOT_WORDS) slot[widx] = (uint32_t)(acc << (32u - nacc));
  }
};

// ---- K7a -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_block_bits(EncodeBatchDev e, int *status) {
  __shared__ EncTablesSmem t;
  load_enc_tables(t, e, blockIdx.y);
  __syncthreads();
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t frame = blockIdx.y;
  __shared__ __align__(16) uint32_t s_rows[128 * ENC_ROW_WORDS];
  stage_cta_blocks(e.quant + (uint64_t)frame * e.nblocks * 64, blockIdx.x * blockDim.x, e.nblocks, s_rows);
  if (blk >= e.nblocks) return;
  const uint32_t *row = s_rows + threadIdx.x * ENC_ROW_WORDS;
  const uint64_t nz = row_nonzero_map(row);
  const int16_t *row16 = reinterpret_cast<const int16_t *>(row);
  int64_t pb = dc_pred_block(e, blk);
  int32_t pred = pb < 0 ? 0 : (int32_t)e.quant[((uint64_t)frame * e.nblocks + pb) * 64];
  const int tsel = e.blk_comp[blk % e.bpm] ? 1 : 0;
  LocalPacker pk;
  pk.init(e.blk_words + ((uint64_t)frame * e.nblocks + blk) * HCJ_ENC_SLOT_WORDS);
  bool ok = encode_block_fields_sparse(nz, [row16](int k) { return (int32_t)row16[k]; }, (int32_t)row16[0] - pred, t.dc[tsel],
                                       t.ac[tsel], pk);
  pk.finish();
  if (!ok) atomicCAS(status + frame, 0, HCJ_ERR_ENCODER_PARAMS);
  e.blk_bits[(uint64_t)frame * (e.nblocks + 1) + blk] = pk.bits;
  if (pk.bits > (uint32_t)HCJ_ENC_SLOT_WORDS * 32u) *e.long_blocks = 1u;  // (every writer stores the same value)
}

// ---- K7o: symbol counts of every frame (HCJ_ENC_OPTIMIZE_HUFFMAN) ----------------------------------
// k_block_bits's grid and staging, block_symbols_sparse instead of the field loop.  counts[frame][4][256]: tables dc 0,
// dc 1, ac 0, ac 1 (Y blocks take table 0, Cb and Cr table 1), zeroed by the chunk's memsets.  Each CTA counts into
// shared memory and adds its non-zero bins to the frame's counts.  The DC size and the EOB, which almost every lane of
// a warp visits at the same point, are summed over the lanes that share the bin before the shared atomic.
__global__ void __launch_bounds__(128) k_symbol_counts(EncodeBatchDev e, uint32_t *counts, int *status) {
  __shared__ uint32_t s_hist[4 * 256];
  __shared__ __align__(16) uint32_t s_rows[128 * ENC_ROW_WORDS];
  for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) s_hist[i] = 0;
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t frame = blockIdx.y;
  stage_cta_blocks(e.quant + (uint64_t)frame * e.nblocks * 64, blockIdx.x * blockDim.x, e.nblocks, s_rows);  // (barrier)
  if (blk < e.nblocks) {
    const uint32_t *row = s_rows + threadIdx.x * ENC_ROW_WORDS;
    const uint64_t nz = row_nonzero_map(row);
    const int16_t *row16 = reinterpret_cast<const int16_t *>(row);
    int64_t pb = dc_pred_block(e, blk);
    int32_t pred = pb < 0 ? 0 : (int32_t)e.quant[((uint64_t)frame * e.nblocks + pb) * 64];
    const int tsel = e.blk_comp[blk % e.bpm] ? 1 : 0;
    bool legal = true;
    auto visit = [&](bool is_ac, uint32_t sym) {
      legal &= annex_k_symbol(is_ac, sym);
      const uint32_t bin = ((is_ac ? 2u : 0u) + tsel) * 256u + sym;
      if (!is_ac || sym == 0x00u) {
        const uint32_t peers = __match_any_sync(__activemask(), bin);
        if ((threadIdx.x & 31u) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(s_hist + bin, (uint32_t)__popc(peers));
      } else {
        atomicAdd(s_hist + bin, 1u);
      }
    };
    const bool ok = block_symbols_sparse(nz, [row16](int k) { return (int32_t)row16[k]; }, (int32_t)row16[0] - pred, visit);
    // a symbol the default tables lack: the status the default encode reports (k_block_bits)
    if (!ok || !legal) atomicCAS(status + frame, 0, HCJ_ERR_ENCODER_PARAMS);
  }
  __syncthreads();
  uint32_t *dst = counts + (uint64_t)frame * 4 * 256;
  for (int i = threadIdx.x; i < 4 * 256; i += blockDim.x) {
    const uint32_t v = s_hist[i];
    if (v) atomicAdd(dst + i, v);
  }
}

// ---- K7t: the optimal tables and the header of every frame (HCJ_ENC_OPTIMIZE_HUFFMAN) -------------------
// One CTA per frame, one warp per table (dc 0, dc 1, ac 0, ac 1; warps 1 and 3 idle for 400).  Each warp runs K.2
// (k2_optimal_table) on its counts and writes the canonical codes into the frame's slot of `tables` ([tab_stride]
// words: dc[2][16], then ac[2][256], the layout of the shared default tables).  Then the CTA writes the frame's header:
// the shared header's bytes before its first DHT segment, the four (two) DHT segments with this frame's tables in the
// same order and with the same class / id bytes, the shared header's bytes after its last DHT segment.
__global__ void __launch_bounds__(128) k_huff_tables(EncodeBatchDev e, const uint32_t *counts, uint32_t *tables, uint8_t *headers,
                                                     uint32_t *header_len, uint32_t dht_off, uint32_t dht_end) {
  __shared__ K2Scratch s_k2[4];
  __shared__ uint8_t s_bits[4][16];
  __shared__ uint8_t s_val[4][256];
  __shared__ int s_nv[4];
  const uint32_t frame = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntab = e.ncomp == 1 ? 1 : 2, cls = warp >> 1, t = warp & 1;
  const bool active = t < ntab;
  if (active) {
    const K2Lanes w{lane, 32};
    const int nv = k2_optimal_table(w, counts + ((uint64_t)frame * 4 + warp) * 256, s_k2[warp], s_bits[warp], s_val[warp]);
    uint32_t *tab = tables + (uint64_t)frame * e.tab_stride;
    uint32_t *codes = cls ? tab + 32 + t * 256 : tab + t * 16;
    for (int i = lane; i < (cls ? 256 : 16); i += 32) codes[i] = 0u;
    __syncwarp();
    if (lane == 0) {
      canonical_codes(s_bits[warp], s_val[warp], cls == 0, codes);
      s_nv[warp] = nv;
    }
  }
  __syncthreads();
  uint8_t *h = headers + (uint64_t)frame * e.frame_header_stride;
  uint32_t seg_off[4], pos = dht_off;
  for (int k = 0; k < 4; k++) {
    seg_off[k] = pos;
    if ((k & 1) < ntab) pos += 21u + (uint32_t)s_nv[k];  // FF C4, length, Tc Th, 16 counts, values (markers.ml:222-231)
  }
  const uint32_t suffix = e.header_len - dht_end;
  for (uint32_t i = threadIdx.x; i < dht_off; i += blockDim.x) h[i] = e.header[i];
  for (uint32_t i = threadIdx.x; i < suffix; i += blockDim.x) h[pos + i] = e.header[dht_end + i];
  if (active) {
    uint8_t *d = h + seg_off[warp];
    const int nv = s_nv[warp], len = 19 + nv;
    for (int i = lane; i < 21 + nv; i += 32)
      d[i] = i == 0 ? 0xffu : i == 1 ? 0xc4u : i == 2 ? (uint8_t)(len >> 8) : i == 3 ? (uint8_t)len : i == 4 ? (uint8_t)((cls << 4) | t)
             : i < 21 ? s_bits[warp][i - 5] : s_val[warp][i - 21];
  }
  if (threadIdx.x == 0) header_len[frame] = pos + suffix;
}

// ---- K7b: in-place exclusive scan of blk_bits per frame; entry [nblocks] receives the total ---------
constexpr int SCAN_THREADS = 1024;
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_bits(EncodeBatchDev e) {
  __shared__ uint32_t s_warp[SCAN_THREADS / 32];  // inclusive sums of the warps, then their exclusive prefix
  __shared__ uint32_t s_total;
  uint32_t *bits = e.blk_bits + (uint64_t)blockIdx.x * (e.nblocks + 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t carry = 0;
  for (uint32_t base = 0; base < e.nblocks; base += SCAN_THREADS) {
    uint32_t i = base + threadIdx.x;
    uint32_t v = i < e.nblocks ? bits[i] : 0;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    // the 32 warp sums are scanned by warp 0 (every thread used to add them up itself: 32 shared-memory reads and 64
    // additions per thread and round)
    if (warp == 0) {
      const uint32_t w = s_warp[lane];
      uint32_t wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += t;
      }
      s_warp[lane] = wi - w;
      if (lane == 31) s_total = wi;
    }
    __syncthreads();
    if (i < e.nblocks) bits[i] = carry + s_warp[warp] + incl - v;
    carry += s_total;
    __syncthreads();  // s_warp / s_total are written again in the next round
  }
  if (threadIdx.x == 0) bits[e.nblocks] = carry;
}

// Segment s of a frame covers blocks [s * ri * bpm, min((s + 1) * ri * bpm, nblocks)).  Its packed bits
// start at byte  floor(P[first] / 8) + s  of the frame's raw buffer (P = exclusive bit prefix): segments
// are byte aligned and never overlap because each one wastes less than a byte of rounding.
__device__ __forceinline__ uint32_t seg_first_block(const EncodeBatchDev &e, uint32_t s) {
  return e.restart_interval ? min(s * e.restart_interval * e.bpm, e.nblocks) : (s ? e.nblocks : 0u);
}

struct BitPacker {
  uint32_t *words;  // big-endian 32-bit words of the raw buffer
  uint64_t acc;     // pending bits, right-aligned
  uint32_t nacc;    // number of pending bits (< 32 between calls)
  uint32_t widx;    // next word to write
  bool first;
  __device__ __forceinline__ void init(uint8_t *raw, uint64_t bitpos) {
    words = reinterpret_cast<uint32_t *>(raw);
    widx = (uint32_t)(bitpos >> 5);
    nacc = (uint32_t)(bitpos & 31u);  // leading bits of the first word belong to the previous block: zeros here
    acc = 0;
    first = true;
  }
  __device__ __forceinline__ void flush_word(uint32_t w) {
    uint32_t le = bswap32(w);
    if (first) {
      atomicOr(words + widx, le);
      first = false;
    } else {
      words[widx] = le;
    }
    widx++;
  }
  __device__ __forceinline__ void operator()(uint32_t bits, uint32_t n) {
    if (n == 0) return;
    acc = (acc << n) | (uint64_t)(bits & ((1u << n) - 1u));
    nacc += n;
    if (nacc >= 32u) {
      nacc -= 32u;
      flush_word((uint32_t)(acc >> nacc));
      acc &= (1ull << nacc) - 1ull;
    }
  }
  __device__ __forceinline__ void finish() {
    if (nacc) {
      uint32_t le = bswap32((uint32_t)(acc << (32u - nacc)));
      atomicOr(words + widx, le);
    }
  }
};

// ---- K7c: every block's bit string goes to its bit offset in the frame's raw buffer -------------------------
// Word j of the destination takes (string word j - 1 : string word j) >> phase; the first and the last word are shared
// with the neighbouring blocks (atomicOr into the zeroed buffer), the words in between are this block's alone.
__global__ void __launch_bounds__(128) k_place(EncodeBatchDev e) {
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t frame = blockIdx.y;
  if (blk >= e.nblocks) return;
  const uint32_t *P = e.blk_bits + (uint64_t)frame * (e.nblocks + 1);
  const uint32_t p0 = P[blk], nb = P[blk + 1] - p0;
  if (nb > (uint32_t)HCJ_ENC_SLOT_WORDS * 32u) return;  // k_pack's
  const uint32_t seg = e.restart_interval ? (blk / e.bpm) / e.restart_interval : 0;
  const uint32_t first = seg_first_block(e, seg), next = seg_first_block(e, seg + 1);
  const uint32_t pf = P[first];
  const uint64_t bitpos = (uint64_t)((pf >> 3) + seg) * 8 + (p0 - pf);
  uint32_t *words = reinterpret_cast<uint32_t *>(e.raw + (uint64_t)frame * e.raw_stride);
  const uint32_t *slot = e.blk_words + ((uint64_t)frame * e.nblocks + blk) * HCJ_ENC_SLOT_WORDS;
  const uint32_t sh = (uint32_t)(bitpos & 31u), nw = (nb + 31u) >> 5, nout = (sh + nb + 31u) >> 5;
  uint32_t *dst = words + (bitpos >> 5);
  uint32_t prev = 0;
  for (uint32_t j = 0; j < nout; j++) {
    const uint32_t cur = j < nw ? slot[j] : 0u;
    const uint32_t le = bswap32(__funnelshift_r(cur, prev, sh));
    prev = cur;
    if (j == 0 || j + 1 == nout) atomicOr(dst + j, le);
    else dst[j] = le;
  }
  if (blk + 1 == next) {  // last block of the segment: flush_with_1s
    const uint32_t pad = (8u - ((P[next] - pf) & 7u)) & 7u;
    if (pad) {
      const uint64_t bp = bitpos + nb;
      const uint32_t sh2 = (uint32_t)(bp & 31u), v = ((1u << pad) - 1u) << (32u - pad);
      atomicOr(words + (bp >> 5), bswap32(v >> sh2));
      if (sh2 + pad > 32u) atomicOr(words + (bp >> 5) + 1, bswap32(v << (32u - sh2)));
    }
  }
}

// ---- K7d: the blocks whose bit string does not fit the slot run the field loop again, straight into the raw buffer ----
__global__ void __launch_bounds__(128) k_pack(EncodeBatchDev e) {
  const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t frame = blockIdx.y;
  const uint32_t *P = e.blk_bits + (uint64_t)frame * (e.nblocks + 1);
  const bool mine = blk < e.nblocks && P[blk + 1] - P[blk] > (uint32_t)HCJ_ENC_SLOT_WORDS * 32u;
  if (!__syncthreads_or(mine)) return;  // CTA-uniform: almost every CTA leaves here
  __shared__ EncTablesSmem t;
  load_enc_tables(t, e, blockIdx.y);
  __syncthreads();
  __shared__ __align__(16) uint32_t s_rows[128 * ENC_ROW_WORDS];
  stage_cta_blocks(e.quant + (uint64_t)frame * e.nblocks * 64, blockIdx.x * blockDim.x, e.nblocks, s_rows);
  if (!mine) return;
  const uint32_t seg = e.restart_interval ? (blk / e.bpm) / e.restart_interval : 0;
  const uint32_t first = seg_first_block(e, seg), next = seg_first_block(e, seg + 1);
  const uint32_t seg_byte = (P[first] >> 3) + seg;
  const uint64_t bitpos = (uint64_t)seg_byte * 8 + (P[blk] - P[first]);

  const uint32_t *row = s_rows + threadIdx.x * ENC_ROW_WORDS;
  const uint64_t nz = row_nonzero_map(row);
  const int16_t *row16 = reinterpret_cast<const int16_t *>(row);
  int64_t pb = dc_pred_block(e, blk);
  int32_t pred = pb < 0 ? 0 : (int32_t)e.quant[((uint64_t)frame * e.nblocks + pb) * 64];
  const int tsel = e.blk_comp[blk % e.bpm] ? 1 : 0;
  BitPacker pk;
  pk.init(e.raw + (uint64_t)frame * e.raw_stride, bitpos);
  encode_block_fields_sparse(nz, [row16](int k) { return (int32_t)row16[k]; }, (int32_t)row16[0] - pred, t.dc[tsel], t.ac[tsel], pk);
  if (blk + 1 == next) {  // last block of the segment: flush_with_1s
    uint32_t segbits = P[next] - P[first];
    uint32_t pad = (8u - (segbits & 7u)) & 7u;
    pk((1u << pad) - 1u, pad);
  }
  pk.finish();
}

// ---- K8a: stuffed size of every segment ------------------------------------------------------------
__device__ __forceinline__ void seg_raw_range(const EncodeBatchDev &e, const uint32_t *P, uint32_t seg, uint32_t &byte0,
                                              uint32_t &nbytes) {
  const uint32_t first = seg_first_block(e, seg), next = seg_first_block(e, seg + 1);
  byte0 = (P[first] >> 3) + seg;
  nbytes = (P[next] - P[first] + 7u) >> 3;
}

// A unit = one warp's share of a segment: the whole segment when restart intervals keep segments short,
// STUFF_CHUNK raw bytes of it otherwise (a scan without restart markers is one segment per frame).
constexpr uint32_t STUFF_CHUNK = 1024;
__device__ __forceinline__ void unit_raw_range(const EncodeBatchDev &e, const uint32_t *P, uint32_t unit, uint32_t &seg,
                                               uint32_t &byte0, uint32_t &nbytes, bool &last_of_seg) {
  seg = unit / e.seg_chunks;
  const uint32_t chunk = unit - seg * e.seg_chunks;
  uint32_t b0, n;
  seg_raw_range(e, P, seg, b0, n);
  last_of_seg = chunk + 1 == e.seg_chunks;
  if (e.seg_chunks > 1) {
    const uint32_t lo = min(chunk * STUFF_CHUNK, n), hi = min(lo + STUFF_CHUNK, n);
    byte0 = b0 + lo;
    nbytes = hi - lo;
  } else {
    byte0 = b0;
    nbytes = n;
  }
}

__global__ void __launch_bounds__(128) k_seg_count(EncodeBatchDev e) {
  const uint32_t unit = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const uint32_t frame = blockIdx.y, lane = threadIdx.x & 31;
  if (unit >= e.nseg * e.seg_chunks) return;
  const uint32_t *P = e.blk_bits + (uint64_t)frame * (e.nblocks + 1);
  uint32_t seg, byte0, nbytes;
  bool last;
  unit_raw_range(e, P, unit, seg, byte0, nbytes, last);
  const uint8_t *raw = e.raw + (uint64_t)frame * e.raw_stride + byte0;
  uint32_t ff = 0;
  for (uint32_t i = lane; i < nbytes; i += 32) ff += raw[i] == 0xffu;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) ff += __shfl_xor_sync(0xffffffffu, ff, s);
  if (lane == 0) e.seg_bytes[(uint64_t)frame * (e.nseg * e.seg_chunks + 1) + unit] = nbytes + ff;
}

// ---- K8b: per frame, exclusive scan of the unit sizes (+2 bytes of RSTn after each segment but the last),
//      starting after the header; copies the header; writes the frame's total length -------------------
__global__ void __launch_bounds__(SCAN_THREADS) k_seg_scan(EncodeBatchDev e) {
  __shared__ uint32_t s_warp[SCAN_THREADS / 32];
  const uint32_t frame = blockIdx.x;
  const uint32_t nunits = e.nseg * e.seg_chunks;
  uint32_t *sb = e.seg_bytes + (uint64_t)frame * (nunits + 1);
  uint8_t *out = e.out + (uint64_t)frame * e.out_stride;
  const uint8_t *header = e.frame_header ? e.frame_header + frame * e.frame_header_stride : e.header;
  const uint32_t header_len = e.frame_header ? e.frame_header_len[frame] : e.header_len;
  for (uint32_t i = threadIdx.x; i < header_len; i += SCAN_THREADS) out[i] = header[i];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t carry = header_len;
  for (uint32_t base = 0; base < nunits; base += SCAN_THREADS) {
    uint32_t i = base + threadIdx.x;
    const bool rst = i < nunits && (i + 1) % e.seg_chunks == 0 && (i + 1) / e.seg_chunks < e.nseg;
    uint32_t v = i < nunits ? sb[i] + (rst ? 2u : 0u) : 0;
    uint32_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t wbase = 0, total = 0;
#pragma unroll
    for (int k = 0; k < SCAN_THREADS / 32; k++) {
      uint32_t t = s_warp[k];
      if (k < warp) wbase += t;
      total += t;
    }
    if (i < nunits) sb[i] = carry + wbase + incl - v;
    carry += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    sb[nunits] = carry;
    out[carry] = 0xff;  // complete_and_write_eoi (encoder.ml:507-510)
    out[carry + 1] = 0xd9;
    e.out_len[frame] = carry + 2;
  }
}

// ---- K8c: copy with byte stuffing; one warp per unit ------------------------------------------------
__global__ void __launch_bounds__(128) k_stuff(EncodeBatchDev e) {
  const uint32_t unit = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const uint32_t frame = blockIdx.y, lane = threadIdx.x & 31;
  const uint32_t nunits = e.nseg * e.seg_chunks;
  if (unit >= nunits) return;
  const uint32_t *P = e.blk_bits + (uint64_t)frame * (e.nblocks + 1);
  const uint32_t *sb = e.seg_bytes + (uint64_t)frame * (nunits + 1);
  uint32_t seg, byte0, nbytes;
  bool last;
  unit_raw_range(e, P, unit, seg, byte0, nbytes, last);
  const uint8_t *raw = e.raw + (uint64_t)frame * e.raw_stride + byte0;
  uint8_t *out = e.out + (uint64_t)frame * e.out_stride;
  uint32_t opos = sb[unit];
  for (uint32_t base = 0; base < nbytes; base += 32 * 8) {  // 8 bytes per lane per round
    uint32_t i0 = base + lane * 8;
    uint8_t v[8];
    uint32_t n = 0, ff = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      bool in = i0 + k < nbytes;
      v[k] = in ? raw[i0 + k] : 0;
      n += in;
      ff += in && v[k] == 0xffu;
    }
    uint32_t cnt = n + ff, incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += t;
    }
    uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    uint32_t o = opos + incl - cnt;
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (i0 + k < nbytes) {
        out[o++] = v[k];
        if (v[k] == 0xffu) out[o++] = 0x00;  // Writer.flush ~stuffing:true (bitstream_writer.ml:25-29)
      }
    opos += total;
  }
  if (lane == 0 && last && seg + 1 < e.nseg) {  // stated extension: RSTn, n = segment index mod 8
    out[opos] = 0xff;
    out[opos + 1] = (uint8_t)(0xd0 + (seg & 7u));
  }
}

// ---- K10 -----------------------------------------------------------------------------------------
// RGB24 frames -> the planar frames k_fdct_quant reads (Frame.input layout: Y of w x h, then Cb and Cr of the chroma
// plane's size; Y only for 400).  The stated forward conversion (rgb_to_ycc_fixed, DESIGN.md 5), then
// Planar_444.convert_to_420 / _422 (planar_444.ml:18-23,68-80) over the ROUNDED 4:4:4 chroma samples: an odd last
// column or row of 4:4:4 chroma is dropped.  A bandwidth kernel like k_rgb_sub_pairs in the other direction: one
// thread per group of 16 pixels (of two rows for 4:2:0, which share their chroma samples), every load issued before any
// arithmetic, 16-byte loads (a row that is not 16-byte aligned is realigned from the aligned chunks around it with
// funnel shifts), alignment-adaptive stores.  Frames come from a device-side pointer table, so uploaded frames and the
// caller's device buffers take the same code.
struct RgbToYcc {
  const uint8_t *const *rgb;  // [frames] w * h * 3 bytes each
  uint8_t *dst;               // [frames][frame_bytes]
  uint64_t frame_bytes, off_cb, off_cr;
  int w, h, cw;               // cw: width of the chroma planes
  uint32_t groups, sets;      // 16-pixel groups per row; row sets (pairs of rows for 4:2:0) per frame
};

// The aligned 16-byte chunks that hold the 48 bytes at p: three when p is 16-byte aligned, four otherwise.  Each chunk
// holds at least one of the 48 bytes, so nothing is read outside the 16-byte granules of the row.
__device__ __forceinline__ void load48_raw(const uint8_t *p, uint32_t (&u)[16]) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint4 *q = reinterpret_cast<const uint4 *>(a & ~(uintptr_t)15);
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const uint4 v = __ldg(q + k);
    u[4 * k] = v.x, u[4 * k + 1] = v.y, u[4 * k + 2] = v.z, u[4 * k + 3] = v.w;
  }
  uint4 v = make_uint4(0u, 0u, 0u, 0u);
  if (a & 15u) v = __ldg(q + 3);
  u[12] = v.x, u[13] = v.y, u[14] = v.z, u[15] = v.w;
}
// The 48 bytes at p as 12 words, from the chunks load48_raw fetched: a word shift by selects, then a byte shift.
__device__ __forceinline__ void align48(const uint8_t *p, const uint32_t (&u)[16], uint32_t (&w)[12]) {
  const uint32_t a = (uint32_t)reinterpret_cast<uintptr_t>(p) & 15u;
  if (a == 0u) {
#pragma unroll
    for (int k = 0; k < 12; k++) w[k] = u[k];
    return;
  }
  const uint32_t q = a >> 2, sh = 8u * (a & 3u);
  uint32_t v[13];
#pragma unroll
  for (int k = 0; k < 13; k++) v[k] = q == 0u ? u[k] : q == 1u ? u[k + 1] : q == 2u ? u[k + 2] : u[k + 3];
#pragma unroll
  for (int k = 0; k < 12; k++) w[k] = __funnelshift_r(v[k], v[k + 1], sh);
}
__device__ __forceinline__ int rgb_byte(const uint32_t (&w)[12], int j) { return (int)__byte_perm(w[j >> 2], 0u, 0x4440u | (j & 3)); }
// byte 2 (the sample, see rgb_to_ycc_fixed) of four sums -> one word
__device__ __forceinline__ uint32_t pack_b2(int t0, int t1, int t2, int t3) {
  return __byte_perm(__byte_perm(t0, t1, 0x0062u), __byte_perm(t2, t3, 0x0062u), 0x5410u);
}
__device__ __forceinline__ uint32_t pack_b0(int c0, int c1, int c2, int c3) {
  return __byte_perm(__byte_perm(c0, c1, 0x0040u), __byte_perm(c2, c3, 0x0040u), 0x5410u);
}

// The short last group of a row (n < 16 pixels, which is where an odd last column lies), and the lone last row of a
// 4:2:0 frame of odd height: byte by byte.
template <int CHROMA>
__device__ __forceinline__ void rgb_to_ycc_tail(const uint8_t *src, int w, int n, bool two, uint8_t *dy, uint8_t *dcb, uint8_t *dcr) {
  const int rows = two ? 2 : 1;
  for (int r = 0; r < rows; r++)
    for (int i = 0; i < n; i++) {
      const uint8_t *p = src + ((size_t)r * w + i) * 3;
      int ty, tcb, tcr;
      rgb_to_ycc_fixed(p[0], p[1], p[2], ty, tcb, tcr);
      dy[(size_t)r * w + i] = (uint8_t)(ty >> 16);
      if (CHROMA == 444) dcb[i] = (uint8_t)(tcb >> 16), dcr[i] = (uint8_t)(tcr >> 16);
    }
  if constexpr (CHROMA == 420 || CHROMA == 422) {
    if (CHROMA == 420 && !two) return;
    for (int j = 0; j < n / 2; j++) {
      int sb = 0, sr = 0;
      for (int r = 0; r < rows; r++)
        for (int i = 2 * j; i < 2 * j + 2; i++) {
          const uint8_t *p = src + ((size_t)r * w + i) * 3;
          int ty, tcb, tcr;
          rgb_to_ycc_fixed(p[0], p[1], p[2], ty, tcb, tcr);
          sb += tcb >> 16, sr += tcr >> 16;
        }
      dcb[j] = (uint8_t)(CHROMA == 420 ? (sb + 2) >> 2 : (sb + 1) >> 1);  // avg4 / avg2 (planar_444.ml:4-16)
      dcr[j] = (uint8_t)(CHROMA == 420 ? (sr + 2) >> 2 : (sr + 1) >> 1);
    }
  }
}

template <int CHROMA>
__global__ void __launch_bounds__(128, 8) k_rgb_to_ycc(RgbToYcc a) {
  constexpr int ROWS = CHROMA == 420 ? 2 : 1;
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, set = t / a.groups, g = t - set * a.groups;
  if (set >= a.sets) return;
  const int x0 = (int)g * 16, y0 = (int)set * ROWS, n = min(16, a.w - x0);
  const bool two = ROWS == 2 && y0 + 1 < a.h;
  const uint8_t *src = a.rgb[blockIdx.y] + ((size_t)y0 * a.w + x0) * 3;
  uint8_t *frame = a.dst + (uint64_t)blockIdx.y * a.frame_bytes;
  uint8_t *dy = frame + (size_t)y0 * a.w + x0;
  uint8_t *dcb = frame + a.off_cb + (size_t)set * a.cw + (CHROMA == 444 ? x0 : x0 / 2), *dcr = dcb + (a.off_cr - a.off_cb);
  if (n < 16 || (ROWS == 2 && !two)) {
    rgb_to_ycc_tail<CHROMA>(src, a.w, n, two, dy, dcb, dcr);
    return;
  }
  uint32_t u0[16], u1[16], w0[12], w1[12];
  load48_raw(src, u0);
  if (ROWS == 2) load48_raw(src + (size_t)a.w * 3, u1);
  align48(src, u0, w0);
  if (ROWS == 2) align48(src + (size_t)a.w * 3, u1, w1);
  uint32_t oy0[4], oy1[4], ocb[4], ocr[4];
  int cb[8], cr[8];
#pragma unroll
  for (int q = 0; q < 4; q++) {  // pixels 4q .. 4q + 3
    int ty[4], tb[4], tr[4], uy[4], ub[4], ur[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int j = 3 * (4 * q + i);
      rgb_to_ycc_fixed(rgb_byte(w0, j), rgb_byte(w0, j + 1), rgb_byte(w0, j + 2), ty[i], tb[i], tr[i]);
      if (ROWS == 2) rgb_to_ycc_fixed(rgb_byte(w1, j), rgb_byte(w1, j + 1), rgb_byte(w1, j + 2), uy[i], ub[i], ur[i]);
    }
    oy0[q] = pack_b2(ty[0], ty[1], ty[2], ty[3]);
    if (ROWS == 2) oy1[q] = pack_b2(uy[0], uy[1], uy[2], uy[3]);
    if (CHROMA == 444) {
      ocb[q] = pack_b2(tb[0], tb[1], tb[2], tb[3]);
      ocr[q] = pack_b2(tr[0], tr[1], tr[2], tr[3]);
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {  // avg4 / avg2 (planar_444.ml:4-16) of the rounded samples
      if (CHROMA == 420) {
        cb[2 * q + k] = ((tb[2 * k] >> 16) + (tb[2 * k + 1] >> 16) + (ub[2 * k] >> 16) + (ub[2 * k + 1] >> 16) + 2) >> 2;
        cr[2 * q + k] = ((tr[2 * k] >> 16) + (tr[2 * k + 1] >> 16) + (ur[2 * k] >> 16) + (ur[2 * k + 1] >> 16) + 2) >> 2;
      } else if (CHROMA == 422) {
        cb[2 * q + k] = ((tb[2 * k] >> 16) + (tb[2 * k + 1] >> 16) + 1) >> 1;
        cr[2 * q + k] = ((tr[2 * k] >> 16) + (tr[2 * k + 1] >> 16) + 1) >> 1;
      }
    }
  }
  store_any<4>(dy, oy0, 16);
  if (ROWS == 2) store_any<4>(dy + a.w, oy1, 16);
  if (CHROMA == 444) {
    store_any<4>(dcb, ocb, 16);
    store_any<4>(dcr, ocr, 16);
  } else if (CHROMA != 400) {
    const uint32_t sb[2] = {pack_b0(cb[0], cb[1], cb[2], cb[3]), pack_b0(cb[4], cb[5], cb[6], cb[7])};
    const uint32_t sr[2] = {pack_b0(cr[0], cr[1], cr[2], cr[3]), pack_b0(cr[4], cr[5], cr[6], cr[7])};
    store_any<2>(dcb, sb, 8);
    store_any<2>(dcr, sr, 8);
  }
}

uint64_t rgb_frame_planar_bytes(int w, int h, int chroma) {  // Frame.create (frame.ml:32-40); one plane for 400
  return chroma == 400 ? (uint64_t)w * h : yuv_frame_bytes(w, h, chroma);
}

void launch_rgb_to_ycc(const uint8_t *const *rgb, int frames, int w, int h, int chroma, uint8_t *dst, cudaStream_t s) {
  if (frames <= 0 || w <= 0 || h <= 0) return;
  RgbToYcc a;
  a.rgb = rgb;
  a.dst = dst;
  a.w = w;
  a.h = h;
  a.cw = chroma == 444 ? w : w / 2;
  const int ch = chroma == 420 ? h / 2 : h;
  a.frame_bytes = rgb_frame_planar_bytes(w, h, chroma);
  a.off_cb = (uint64_t)w * h;
  a.off_cr = a.off_cb + (uint64_t)a.cw * ch;
  a.groups = (uint32_t)((w + 15) / 16);
  a.sets = (uint32_t)(chroma == 420 ? (h + 1) / 2 : h);
  const dim3 grid((unsigned)(((uint64_t)a.groups * a.sets + 127) / 128), (unsigned)frames);
  switch (chroma) {
    case 420: k_rgb_to_ycc<420><<<grid, 128, 0, s>>>(a); break;
    case 422: k_rgb_to_ycc<422><<<grid, 128, 0, s>>>(a); break;
    case 444: k_rgb_to_ycc<444><<<grid, 128, 0, s>>>(a); break;
    default: k_rgb_to_ycc<400><<<grid, 128, 0, s>>>(a); break;
  }
}

void launch_encode(const EncodeBatchDev &e, cudaStream_t s) {
  if (e.n == 0) return;
  dim3 gb((e.nblocks + 127) / 128, e.n);
  k_fdct_quant<<<gb, 128, 0, s>>>(e);
}

// k_fdct_quant, k_block_bits, k_scan_bits, k_gather_totals, k_place, k_seg_count, k_seg_scan, k_stuff (+ k_pack for chunks with
// long blocks; + k_symbol_counts and k_huff_tables with HCJ_ENC_OPTIMIZE_HUFFMAN)
int encode_kernel_count() { return 8; }

// Gathers the per-frame totals of the bit scan into a dense array for one small D2H copy.
__global__ void k_gather_totals(EncodeBatchDev e, uint32_t *totals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < e.n) totals[i] = e.blk_bits[(uint64_t)i * (e.nblocks + 1) + e.nblocks];
}

static void launch_bit_lengths(const EncodeBatchDev &e, int *d_status, uint32_t *d_totals, cudaStream_t s) {
  dim3 gb((e.nblocks + 127) / 128, e.n);
  k_block_bits<<<gb, 128, 0, s>>>(e, d_status);
  k_scan_bits<<<e.n, SCAN_THREADS, 0, s>>>(e);
  k_gather_totals<<<(e.n + 127) / 128, 128, 0, s>>>(e, d_totals);
}

// HCJ_ENC_OPTIMIZE_HUFFMAN: per-frame symbol counts, tables and headers, between k_fdct_quant and k_block_bits
struct HuffOpt {
  uint32_t *counts;      // [n][4][256], zeroed before every chunk
  uint32_t *tables;      // [n][e.tab_stride]
  uint8_t *headers;      // [n][e.frame_header_stride]
  uint32_t *header_len;  // [n]
  uint32_t dht_off, dht_end;  // the DHT segments of the shared header: bytes [dht_off, dht_end)
};
static void launch_huff_opt(const EncodeBatchDev &e, const HuffOpt &o, int *d_status, cudaStream_t s) {
  dim3 gb((e.nblocks + 127) / 128, e.n);
  k_symbol_counts<<<gb, 128, 0, s>>>(e, o.counts, d_status);
  k_huff_tables<<<e.n, 128, 0, s>>>(e, o.counts, o.tables, o.headers, o.header_len, o.dht_off, o.dht_end);
}

static void launch_entropy(const EncodeBatchDev &e, bool long_blocks, cudaStream_t s) {
  dim3 gb((e.nblocks + 127) / 128, e.n);
  k_place<<<gb, 128, 0, s>>>(e);
  if (long_blocks) k_pack<<<gb, 128, 0, s>>>(e);  // (0.1 ms per 512 x 1080p even when every CTA leaves at once)
  dim3 gs((e.nseg * e.seg_chunks + 3) / 4, e.n);
  k_seg_count<<<gs, 128, 0, s>>>(e);
  k_seg_scan<<<e.n, SCAN_THREADS, 0, s>>>(e);
  k_stuff<<<gs, 128, 0, s>>>(e);
}

// ---- debug tap: Encoder.Block.t of encode_seq (encoder.ml:56-66,195-205,476-505) -------------------
// One thread per block; reads the quantised blocks k_fdct_quant has written (for the DC predictor) and recomputes
// everything else of the block with the model's arithmetic, reconstruction included (Block.decoded, `-verbose`).
struct EncodeBlockLog {  // = hcj_encoder_block (include/hcjpeg.h)
  int32_t x_pos, y_pos, dc_pred, component, nrle;
  uint8_t input_pixels[64];
  int32_t fdct[64];
  int16_t quant[64];
  int16_t rle_run[64], rle_value[64];
  int32_t dequant[64], idct[64];
  uint8_t recon[64], error[64];
};
__global__ void k_encode_block_log(EncodeBatchDev e, uint32_t first, uint32_t count, EncodeBlockLog *out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const uint32_t blk = first + t;
  const uint32_t mcu = blk / e.bpm, k = blk - mcu * e.bpm;
  const int c = e.blk_comp[k];
  const int my = mcu / e.mcus_wide, mx = mcu - my * e.mcus_wide;
  const int x0 = (mx * e.hs[c] + e.blk_bx[k]) * 8, y0 = (my * e.vs[c] + e.blk_by[k]) * 8;  // encoder.ml:486-489
  const uint8_t *src = e.src + e.src_off[c];
  const int sw = e.src_w[c], sh = e.src_h[c], pw = e.plane_w[c];
  const int64_t nsrc = (int64_t)sw * sh;
  EncodeBlockLog &o = out[t];
  o.x_pos = x0;
  o.y_pos = y0;
  o.component = c;
  int32_t v[64];
  for (int y = 0; y < 8; y++)
    for (int x = 0; x < 8; x++) {  // level_shifted_input_block over the zero-initialised padded plane (encoder.ml:81-90)
      int p;
      if (e.linear_blit) {  // encode_monochrome: Plane.blit is one linear copy (encoder.ml:548, plane.ml:20)
        const int64_t at = (int64_t)(y0 + y) * pw + (x0 + x);
        p = at < nsrc ? (int)src[at] : 0;
      } else {
        p = (x0 + x < sw && y0 + y < sh) ? (int)src[(size_t)(y0 + y) * sw + x0 + x] : 0;
      }
      o.input_pixels[y * 8 + x] = (uint8_t)p;
      v[y * 8 + x] = p - 128;
    }
  fdct_8x8(v);
  const uint16_t *qt = e.qt + (c ? 64 : 0);
  const uint32_t *qr = e.qrecip + (c ? 64 : 0);
  int32_t q[64];
  for (int i = 0; i < 64; i++) {
    o.fdct[i] = v[i];
    const int z = zigzag_forward(i);  // encoder.ml:103-108
    q[z] = quantize(v[i], qt[z], qr[z]);
  }
  for (int z = 0; z < 64; z++) o.quant[z] = (int16_t)q[z];
  // rle (encoder.ml:127-141): the DC differential first, position 63 always emitted
  const int64_t pb = dc_pred_block(e, blk);
  const int32_t pred = pb < 0 ? 0 : (int32_t)e.quant[(uint64_t)pb * 64];
  int n = 0, run = 0;
  o.rle_run[n] = 0;
  o.rle_value[n++] = (int16_t)(q[0] - pred);
  for (int pos = 1; pos < 64; pos++) {
    if (pos == 63 || q[pos] != 0) {
      o.rle_run[n] = (int16_t)run;
      o.rle_value[n++] = (int16_t)q[pos];
      run = 0;
    } else {
      run++;
    }
  }
  o.nrle = n;
  for (int i = n; i < 64; i++) o.rle_run[i] = o.rle_value[i] = 0;
  o.dc_pred = q[0];
  // Block.decoded (encoder.ml:110-125): dequant, idct, recon, error
  int64_t w[64];
  for (int z = 0; z < 64; z++) w[zigzag_inverse(z)] = (int64_t)q[z] * qt[z];
  for (int i = 0; i < 64; i++) o.dequant[i] = (int32_t)w[i];
  idct_8x8<int64_t>(w);
  for (int i = 0; i < 64; i++) {
    o.idct[i] = (int32_t)w[i];
    const int64_t r = w[i] + 128 < 0 ? 0 : w[i] + 128 > 255 ? 255 : w[i] + 128;
    o.recon[i] = (uint8_t)r;
    const int d = (int)r - (int)o.input_pixels[i];
    o.error[i] = (uint8_t)(d < 0 ? -d : d);
  }
}
void launch_encode_block_log(const EncodeBatchDev &e, uint32_t first, uint32_t count, void *out, cudaStream_t s) {
  if (count) k_encode_block_log<<<(count + 63) / 64, 64, 0, s>>>(e, first, count, reinterpret_cast<EncodeBlockLog *>(out));
}

}  // namespace hcjk

// ================================================================================================
// C ABI
// ================================================================================================
namespace {

struct EncodeSetup {
  hcj::EncodePlan plan;
  hcjk::EncodeBatchDev dev;
  std::vector<void *> owned;
  std::vector<uint8_t> header;
  int *d_status = nullptr;
};

int setup_encode(hcj_ctx *c, int n, int width, int height, int chroma, int quality, int restart_interval, bool entropy,
                 EncodeSetup *S) {
  int st = hcj::plan_encode(width, height, chroma, quality, restart_interval, &S->plan);
  if (st != HCJ_OK) return st;
  const hcj::EncodePlan &p = S->plan;
  hcjk::EncodeBatchDev &e = S->dev;
  memset(&e, 0, sizeof(e));
  e.n = n;
  e.ncomp = p.ncomp;
  e.bpm = p.bpm;
  uint64_t off = 0;
  e.linear_blit = chroma == 400 ? 1 : 0;
  for (int i = 0; i < p.ncomp; i++) {
    e.hs[i] = p.hs[i];
    e.vs[i] = p.vs[i];
    e.plane_w[i] = p.plane_w[i];
    e.plane_h[i] = p.plane_h[i];
    e.src_w[i] = p.src_w[i];
    e.src_h[i] = p.src_h[i];
    e.src_off[i] = off;
    off += (uint64_t)p.src_w[i] * p.src_h[i];
  }
  e.frame_bytes = off;
  e.mcus_wide = p.mcus_wide;
  e.mcus_high = p.mcus_high;
  e.nblocks = (uint32_t)p.nblocks;
  e.restart_interval = (uint32_t)restart_interval;
  uint32_t nmcu = (uint32_t)(p.mcus_wide * p.mcus_high);
  e.nseg = restart_interval ? (nmcu + restart_interval - 1) / restart_interval : 1;
  for (int k = 0; k < p.bpm; k++) {
    e.blk_comp[k] = (uint8_t)p.blk_comp[k];
    e.blk_bx[k] = (uint8_t)p.blk_bx[k];
    e.blk_by[k] = (uint8_t)p.blk_by[k];
  }
  hcj::write_headers(p, &S->header);
  e.header_len = (uint32_t)S->header.size();

  std::vector<uint32_t> tables(64 * 2 + 32 + 512);
  uint16_t qt16[128];
  for (int t = 0; t < 2; t++)
    for (int i = 0; i < 64; i++) {
      qt16[t * 64 + i] = p.qt[t][i];
      tables[t * 64 + i] = (uint32_t)((1ull << 32) / (4u * p.qt[t][i])) + 1u;  // reciprocal of 4q
    }
  hcj::encoder_tables(0, 2, &tables[128], &tables[160]);
  hcj::encoder_tables(1, 3, &tables[144], &tables[160 + 256]);

  auto alloc = [&](void **ptr, size_t bytes) {
    if (st != HCJ_OK) return;
    st = c->alloc(ptr, bytes);
    if (st == HCJ_OK) S->owned.push_back(*ptr);
  };
  void *d_tables = nullptr, *d_qt = nullptr, *d_hdr = nullptr;
  alloc(&d_tables, tables.size() * 4);
  alloc(&d_qt, sizeof(qt16));
  alloc(&d_hdr, S->header.size() + 16);
  alloc((void **)&e.src, e.frame_bytes * (uint64_t)n + 16);
  alloc((void **)&e.quant, (uint64_t)n * e.nblocks * 128 + 16);
  alloc((void **)&S->d_status, 4 * (size_t)std::max(n, 1));
  if (entropy) {
    alloc((void **)&e.blk_bits, (uint64_t)n * (e.nblocks + 1) * 4);
    alloc((void **)&e.blk_words, (uint64_t)n * e.nblocks * hcjk::HCJ_ENC_SLOT_WORDS * 4);
    alloc((void **)&e.out_len, 4 * (size_t)std::max(n, 1) + 4);
    if (st == HCJ_OK) e.long_blocks = e.out_len + std::max(n, 1);  // one flag behind the lengths
  }
  if (st != HCJ_OK) return st;
  e.qrecip = reinterpret_cast<const uint32_t *>(d_tables);
  e.dc_codes = e.qrecip + 128;
  e.ac_codes = e.qrecip + 160;
  e.qt = reinterpret_cast<const uint16_t *>(d_qt);
  e.header = reinterpret_cast<const uint8_t *>(d_hdr);
  CU_TRY(cudaMemcpyAsync(d_tables, tables.data(), tables.size() * 4, cudaMemcpyHostToDevice, c->stream));
  CU_TRY(cudaMemcpyAsync(d_qt, qt16, sizeof(qt16), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(cudaMemcpyAsync(d_hdr, S->header.data(), S->header.size(), cudaMemcpyHostToDevice, c->stream));
  CU_TRY(cudaMemsetAsync(S->d_status, 0, 4 * (size_t)std::max(n, 1), c->stream));
  CU_TRY(cudaStreamSynchronize(c->stream));  // `tables` / `qt16` are stack / local storage
  return HCJ_OK;
}

void teardown_encode(hcj_ctx *c, EncodeSetup *S) {
  cudaStreamSynchronize(c->stream);
  for (void *p : S->owned) c->release(p);
  S->owned.clear();
}

}  // namespace

extern "C" {

/* The scalar helpers of the model, evaluated on the host by the very functions the kernels call (hcj_device.cuh). */
int hcj_mag(int cat, int code) {  // Decoder.For_testing.mag' (decoder.ml:73-79)
  if (cat <= 0 || cat > 16) return 0;
  return (int)hcjdev::extend((uint32_t)code & ((1u << cat) - 1u), (uint32_t)cat);
}
int hcj_size(int value) { return (int)hcjdev::coef_size((int32_t)value); }  // Encoder.size (encoder.ml:143)
int hcj_magnitude(int size, int value) {  // Encoder.magnitude (encoder.ml:145-147)
  return (int)hcjdev::coef_magnitude((int32_t)value, (uint32_t)size);
}

int hcj_quant_scale(int chroma_table, int quality, uint16_t out[64]) {  // Quant_tables.scale (quant_tables.ml:139-147)
  if (!out) return HCJ_ERR_INVALID_ARG;
  hcj::quant_scale(chroma_table != 0, quality, out);
  return HCJ_OK;
}
int hcj_encoder_code(int table, int run, int size, int *bits, int *length) {  // Tables.Encoder.dc_table / ac_table (tables.ml:504-545)
  if (table < 0 || table > 3 || run < 0 || run > 15 || size < 0 || size > 15 || !bits || !length) return HCJ_ERR_INVALID_ARG;
  uint32_t dc[16], ac[256];
  hcj::encoder_tables(table & 1, 2 + (table & 1), dc, ac);  // exactly what setup_encode uploads for the kernels
  const uint32_t e = table < 2 ? (run == 0 ? dc[size] : 0u) : ac[(run << 4) | size];
  *bits = (int)(e >> 8);
  *length = (int)(e & 0xffu);  // 0: no such code
  return HCJ_OK;
}

size_t hcj_encode_bound(int width, int height, int chroma) {
  hcj::EncodePlan p;
  if (hcj::plan_encode(width, height, chroma, 75, 0, &p) != HCJ_OK) return 0;
  return 1024 + (size_t)p.nblocks * 432 + 16;  // header + 2 x 216 bytes per block (all bytes stuffed) + EOI
}

int hcj_encode_count_kernels(void) { return hcjk::encode_kernel_count(); }

int hcj_write_headers(int width, int height, int chroma, int quality, int restart_interval, uint8_t *out, size_t capacity,
                      size_t *len) {
  if (!out || !len) return HCJ_ERR_INVALID_ARG;
  hcj::EncodePlan p;
  int st = hcj::plan_encode(width, height, chroma, quality, restart_interval, &p);
  if (st != HCJ_OK) return st;
  std::vector<uint8_t> h;
  hcj::write_headers(p, &h);
  *len = h.size();
  if (h.size() > capacity) return HCJ_ERR_BUFFER_TOO_SMALL;
  memcpy(out, h.data(), h.size());
  return HCJ_OK;
}

}  // extern "C"

namespace {

// Where the frames of a chunk come from: the only stage in which the encode entry points differ.
enum class EncodeSource {
  YUV_HOST,    // planar frames in host memory: uploaded into the chunk's slot, which k_fdct_quant reads
  RGB_HOST,    // RGB24 frames in host memory: uploaded into the chunk's slot, converted by k_rgb_to_ycc into e.src
  RGB_DEVICE,  // RGB24 frames in device memory: converted by k_rgb_to_ycc straight from the caller's buffers into e.src
};

// Frames go through the device in chunks: while the kernels of chunk k run, the frames of chunk k + 1 go up on a second
// stream and the files of chunk k - 1 come down on a third (the call used to be H2D, then kernels, then D2H: 41.8 ms per
// 512 x 1080p frames, of which 29 ms is the 1.6 GB of frames on the PCIe link).  The host waits twice per chunk for the
// kernel stream only - for the bit totals that size the byte buffers, and for the file lengths - which the copies on
// the other two streams do not notice.  Uploaded frames and finished files are double-buffered on the device.
int encode_frames(hcj_ctx *c, EncodeSource kind, const uint8_t *const *yuv, int n, int width, int height, int chroma, int quality,
                  int restart_interval, bool optimize, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                  int *status) {
  CU_TRY(cudaSetDevice(c->device));
  int chunk = 64;
  if (const char *ev = getenv("HCJ_ENC_CHUNK")) chunk = std::max(1, atoi(ev));
  const int ch = std::max(1, std::min(n, chunk)), nchunks = n ? (n + ch - 1) / ch : 0;
  EncodeSetup S;
  int st = setup_encode(c, ch, width, height, chroma, quality, restart_interval, true, &S);
  if (st != HCJ_OK) {
    teardown_encode(c, &S);
    return st;
  }
  hcjk::EncodeBatchDev &e = S.dev;
  cudaStream_t s = c->stream, us = c->up_stream ? c->up_stream : c->stream, cs = c->copy_stream ? c->copy_stream : c->stream;
  cudaError_t err = cudaSuccess;
  c->enc_timed = false;
  c->enc_ms = 0.f;
  // upload slots: planar frames go straight into e.src and a second slot, RGB frames into two slots of their own in
  // front of the conversion (whose planar output e.src only the kernel stream touches); slots of finished files grow on
  // demand
  const bool rgb = kind != EncodeSource::YUV_HOST;
  const uint64_t slot_frame = kind == EncodeSource::YUV_HOST ? e.frame_bytes : 3ull * width * height;
  uint8_t *src_slot[2] = {kind == EncodeSource::YUV_HOST ? const_cast<uint8_t *>(e.src) : nullptr, nullptr};
  uint8_t *out_slot[2] = {nullptr, nullptr};
  uint64_t out_cap[2] = {0, 0}, raw_cap = 0, segb_cap = 0;
  auto alloc_owned = [&](void **ptr, size_t bytes) {
    if (st != HCJ_OK) return;
    st = c->alloc(ptr, bytes);
    if (st == HCJ_OK) S.owned.push_back(*ptr);
  };
  if (kind == EncodeSource::RGB_HOST) alloc_owned((void **)&src_slot[0], slot_frame * (uint64_t)ch + 16);
  if (kind != EncodeSource::RGB_DEVICE) {
    if (nchunks > 1) alloc_owned((void **)&src_slot[1], slot_frame * (uint64_t)ch + 16);
    else src_slot[1] = src_slot[0];
  }
  // HCJ_ENC_OPTIMIZE_HUFFMAN: counts, tables and headers of one chunk (the kernel stream runs the chunks one after the
  // other, so one set serves them all); the frames' headers are never longer than the shared one, which sizes out_stride
  hcjk::HuffOpt opt = {};
  if (optimize) {
    const std::vector<uint8_t> &hd = S.header;
    uint32_t p = 2;  // after SOI: segments up to the first DHT, then the DHT segments
    while (p + 4 <= hd.size() && hd[p + 1] != 0xc4) p += 2 + ((hd[p + 2] << 8) | hd[p + 3]);
    opt.dht_off = p;
    while (p + 4 <= hd.size() && hd[p + 1] == 0xc4) p += 2 + ((hd[p + 2] << 8) | hd[p + 3]);
    opt.dht_end = p;
    e.tab_stride = 32 + 512;
    e.frame_header_stride = hcj::align_up(e.header_len, 16);
    alloc_owned((void **)&opt.counts, (uint64_t)ch * 4 * 256 * 4);
    alloc_owned((void **)&opt.tables, (uint64_t)ch * e.tab_stride * 4);
    alloc_owned((void **)&opt.headers, (uint64_t)ch * e.frame_header_stride);
    alloc_owned((void **)&opt.header_len, 4 * (uint64_t)ch);
    e.dc_codes = opt.tables;
    e.ac_codes = opt.tables + 32;
    e.frame_header = opt.headers;
    e.frame_header_len = opt.header_len;
  }
  // k_rgb_to_ycc's frame table: the frames of both slots, or every caller frame (chunk k reads entries k * ch ..)
  const uint8_t **d_frames = nullptr;
  std::vector<const uint8_t *> frames;
  if (rgb && st == HCJ_OK) {
    if (kind == EncodeSource::RGB_HOST)
      for (int k = 0; k < 2; k++)
        for (int i = 0; i < ch; i++) frames.push_back(src_slot[k] + (uint64_t)i * slot_frame);
    else
      frames.assign(yuv, yuv + n);
    alloc_owned((void **)&d_frames, frames.size() * sizeof(frames[0]));
    if (st == HCJ_OK && cudaMemcpyAsync(d_frames, frames.data(), frames.size() * sizeof(frames[0]), cudaMemcpyHostToDevice, c->stream) != cudaSuccess)
      st = HCJ_ERR_CUDA - (int)cudaGetLastError();
  }
  std::vector<cudaEvent_t> ev_up(nchunks), ev_src_free(nchunks), ev_done(nchunks), ev_down(nchunks), ev_t(4 * (size_t)nchunks);
  for (auto *v : {&ev_up, &ev_src_free, &ev_done, &ev_down})
    for (auto &x : *v)
      if (err == cudaSuccess) err = cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
  for (auto &x : ev_t)
    if (err == cudaSuccess) err = cudaEventCreate(&x);
  std::vector<uint32_t> lens(std::max(ch, 1));
  std::vector<int> dev_status(std::max(ch, 1), 0);
  auto upload = [&](int k) {  // frames of chunk k -> their slot, behind the kernels that last read it
    const int lo = k * ch, hi = std::min(n, lo + ch);
    if (k >= 2 && err == cudaSuccess) err = cudaStreamWaitEvent(us, ev_src_free[k - 2], 0);
    for (int i = lo; i < hi && err == cudaSuccess && kind != EncodeSource::RGB_DEVICE;) {  // frames that lie back to back in host memory go up as one copy
      int j = i + 1;
      while (j < hi && yuv[j] == yuv[j - 1] + slot_frame) j++;
      err = cudaMemcpyAsync(src_slot[k & 1] + (uint64_t)(i - lo) * slot_frame, yuv[i], slot_frame * (uint64_t)(j - i), cudaMemcpyHostToDevice, us);
      i = j;
    }
    if (err == cudaSuccess) err = cudaEventRecord(ev_up[k], us);
  };
  if (st == HCJ_OK && nchunks > 0) upload(0);
  for (int k = 0; k < nchunks && err == cudaSuccess && st == HCJ_OK; k++) {
    const int lo = k * ch, hi = std::min(n, lo + ch), m = hi - lo;
    if (k + 1 < nchunks) upload(k + 1);
    e.n = m;
    if (!rgb) e.src = src_slot[k & 1];
    // phase 1: coefficients and the bit length of every block; the totals size the byte buffers
    if (err == cudaSuccess) err = cudaStreamWaitEvent(s, ev_up[k], 0);
    if (err == cudaSuccess) err = cudaMemsetAsync(S.d_status, 0, 4 * (size_t)m, s);
    if (err == cudaSuccess) err = cudaMemsetAsync(e.long_blocks, 0, 4, s);
    if (optimize && err == cudaSuccess) err = cudaMemsetAsync(opt.counts, 0, (size_t)m * 4 * 256 * 4, s);
    cudaEventRecord(ev_t[4 * k + 0], s);
    if (rgb)
      hcjk::launch_rgb_to_ycc(d_frames + (kind == EncodeSource::RGB_HOST ? (k & 1) * ch : lo), m, width, height, chroma,
                              const_cast<uint8_t *>(e.src), s);
    hcjk::launch_encode(e, s);
    if (optimize) hcjk::launch_huff_opt(e, opt, S.d_status, s);
    hcjk::launch_bit_lengths(e, S.d_status, e.out_len, s);
    cudaEventRecord(ev_t[4 * k + 1], s);
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaEventRecord(ev_src_free[k], s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(lens.data(), e.out_len, 4 * (size_t)m, cudaMemcpyDeviceToHost, s);
    uint32_t long_blocks = 1;
    if (err == cudaSuccess) err = cudaMemcpyAsync(&long_blocks, e.long_blocks, 4, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaStreamSynchronize(s);
    if (err != cudaSuccess) break;
    uint64_t max_bits = 0;
    for (int i = 0; i < m; i++) max_bits = std::max<uint64_t>(max_bits, lens[i]);
    e.raw_stride = hcj::align_up(max_bits / 8 + e.nseg + 64, 256);
    e.out_stride = hcj::align_up(e.header_len + 2 * e.raw_stride + 2ull * e.nseg + 16, 256);  // every byte stuffed
    e.seg_chunks = e.nseg == 1 ? (uint32_t)((e.raw_stride + hcjk::STUFF_CHUNK - 1) / hcjk::STUFF_CHUNK) : 1u;
    auto ensure = [&](uint8_t **ptr, uint64_t *cap, uint64_t bytes) {  // grow-only workspace (the old block goes back to the pool)
      if (st != HCJ_OK || *cap >= bytes) return;
      void *p = nullptr;
      st = c->alloc(&p, bytes + bytes / 4);
      if (st != HCJ_OK) return;
      S.owned.push_back(p);  // (the smaller block stays owned until teardown: nothing in flight may lose its memory)
      *ptr = static_cast<uint8_t *>(p);
      *cap = bytes + bytes / 4;
    };
    uint8_t *segb = reinterpret_cast<uint8_t *>(e.seg_bytes);
    ensure(&e.raw, &raw_cap, (uint64_t)m * e.raw_stride);
    ensure(&segb, &segb_cap, (uint64_t)m * ((uint64_t)e.nseg * e.seg_chunks + 1) * 4);
    e.seg_bytes = reinterpret_cast<uint32_t *>(segb);
    ensure(&out_slot[k & 1], &out_cap[k & 1], (uint64_t)m * e.out_stride);
    if (st != HCJ_OK) break;
    e.out = out_slot[k & 1];
    // phase 2: pack, stuff, assemble (behind the copies that still read this slot of files)
    if (k >= 2) err = cudaStreamWaitEvent(s, ev_down[k - 2], 0);
    if (err == cudaSuccess) err = cudaMemsetAsync(e.raw, 0, (uint64_t)m * e.raw_stride, s);  // the packer ORs into zeroed words
    cudaEventRecord(ev_t[4 * k + 2], s);
    hcjk::launch_entropy(e, long_blocks != 0, s);
    cudaEventRecord(ev_t[4 * k + 3], s);
    if (err == cudaSuccess) err = cudaGetLastError();
    if (err == cudaSuccess) err = cudaMemcpyAsync(lens.data(), e.out_len, 4 * (size_t)m, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaMemcpyAsync(dev_status.data(), S.d_status, 4 * (size_t)m, cudaMemcpyDeviceToHost, s);
    if (err == cudaSuccess) err = cudaEventRecord(ev_done[k], s);
    if (err == cudaSuccess) err = cudaStreamSynchronize(s);
    if (err == cudaSuccess) err = cudaStreamWaitEvent(cs, ev_done[k], 0);
    for (int i = 0; i < m && err == cudaSuccess; i++) {
      int sti = dev_status[i];
      out_len[lo + i] = lens[i];
      if (sti == HCJ_OK && (!out[lo + i] || out_capacity[lo + i] < lens[i])) sti = HCJ_ERR_BUFFER_TOO_SMALL;
      if (sti == HCJ_OK) err = cudaMemcpyAsync(out[lo + i], e.out + (uint64_t)i * e.out_stride, lens[i], cudaMemcpyDeviceToHost, cs);
      if (status) status[lo + i] = sti;
    }
    if (err == cudaSuccess) err = cudaEventRecord(ev_down[k], cs);
    float a = 0.f, b2 = 0.f;  // kernel time of the chunk (both phases; the host's sizing step in between is not device work)
    if (err == cudaSuccess && cudaEventElapsedTime(&a, ev_t[4 * k], ev_t[4 * k + 1]) == cudaSuccess &&
        cudaEventElapsedTime(&b2, ev_t[4 * k + 2], ev_t[4 * k + 3]) == cudaSuccess)
      c->enc_ms += a + b2;
  }
  // nothing may still be reading the caller's frames or writing the caller's buffers when the call returns
  cudaStreamSynchronize(us);
  cudaStreamSynchronize(cs);
  cudaStreamSynchronize(s);
  c->enc_timed = err == cudaSuccess && st == HCJ_OK && n > 0;
  for (auto *v : {&ev_up, &ev_src_free, &ev_done, &ev_down, &ev_t})
    for (auto &x : *v)
      if (x) cudaEventDestroy(x);
  teardown_encode(c, &S);
  if (st != HCJ_OK) return st;
  return err == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)err;
}

}  // namespace

extern "C" {

int hcj_encode_batch(hcj_ctx *c, const uint8_t *const *yuv, int n, int width, int height, int chroma, int quality,
                     int restart_interval, uint8_t *const *out, const size_t *out_capacity, size_t *out_len, int *status) {
  if (!c || n < 0 || n > HCJ_MAX_BATCH || (n > 0 && (!yuv || !out || !out_capacity || !out_len))) return HCJ_ERR_INVALID_ARG;
  return encode_frames(c, EncodeSource::YUV_HOST, yuv, n, width, height, chroma, quality, restart_interval, false, out, out_capacity,
                       out_len, status);
}

int hcj_encode_batch_ex(hcj_ctx *c, const uint8_t *const *yuv, int n, int width, int height, int chroma, int quality,
                        int restart_interval, unsigned flags, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                        int *status) {
  if (flags & ~HCJ_ENC_OPTIMIZE_HUFFMAN) return HCJ_ERR_INVALID_ARG;
  if (!c || n < 0 || n > HCJ_MAX_BATCH || (n > 0 && (!yuv || !out || !out_capacity || !out_len))) return HCJ_ERR_INVALID_ARG;
  return encode_frames(c, EncodeSource::YUV_HOST, yuv, n, width, height, chroma, quality, restart_interval,
                       (flags & HCJ_ENC_OPTIMIZE_HUFFMAN) != 0, out, out_capacity, out_len, status);
}

int hcj_encode_rgb_batch(hcj_ctx *c, const uint8_t *const *rgb, int n, int width, int height, int chroma, int quality,
                         int restart_interval, unsigned flags, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                         int *status) {
  if (!c || n < 0 || n > HCJ_MAX_BATCH || (n > 0 && (!rgb || !out || !out_capacity || !out_len))) return HCJ_ERR_INVALID_ARG;
  if (flags & ~(HCJ_ENC_SRC_DEVICE | HCJ_ENC_OPTIMIZE_HUFFMAN)) return HCJ_ERR_INVALID_ARG;
  if (flags & HCJ_ENC_SRC_DEVICE) {  // every frame must be device (or managed) memory of the context's device
    for (int i = 0; i < n; i++) {
      cudaPointerAttributes at;
      if (!rgb[i] || cudaPointerGetAttributes(&at, rgb[i]) != cudaSuccess) {
        (void)cudaGetLastError();
        return HCJ_ERR_INVALID_ARG;
      }
      if ((at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) || at.device != c->device) return HCJ_ERR_INVALID_ARG;
    }
  }
  return encode_frames(c, (flags & HCJ_ENC_SRC_DEVICE) ? EncodeSource::RGB_DEVICE : EncodeSource::RGB_HOST, rgb, n, width, height,
                       chroma, quality, restart_interval, (flags & HCJ_ENC_OPTIMIZE_HUFFMAN) != 0, out, out_capacity, out_len, status);
}

int hcj_rgb_to_yuv(hcj_ctx *c, const uint8_t *rgb, int width, int height, int chroma, uint8_t *dst, size_t dst_capacity) {
  if (!c || !rgb || !dst || width < 1 || height < 1 || (chroma != 420 && chroma != 422 && chroma != 444 && chroma != 400))
    return HCJ_ERR_INVALID_ARG;
  const uint64_t nin = 3ull * width * height, nout = hcjk::rgb_frame_planar_bytes(width, height, chroma);
  if (dst_capacity < nout) return HCJ_ERR_BUFFER_TOO_SMALL;
  CU_TRY(cudaSetDevice(c->device));
  void *d_in = nullptr, *d_out = nullptr, *d_tab = nullptr;
  int st = c->alloc(&d_in, nin + 16);
  if (st == HCJ_OK) st = c->alloc(&d_out, nout + 16);
  if (st == HCJ_OK) st = c->alloc(&d_tab, sizeof(void *));
  cudaError_t e = cudaSuccess;
  if (st == HCJ_OK) {
    e = cudaMemcpyAsync(d_in, rgb, nin, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab, &d_in, sizeof(void *), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
      hcjk::launch_rgb_to_ycc(static_cast<const uint8_t *const *>(d_tab), 1, width, height, chroma, static_cast<uint8_t *>(d_out), c->stream);
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(dst, d_out, nout, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
  }
  cudaStreamSynchronize(c->stream);  // nothing in flight may lose its memory
  c->release(d_in);
  c->release(d_out);
  c->release(d_tab);
  if (st != HCJ_OK) return st;
  return e == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)e;
}

// The encoder mirror of hcj_decode_batch_multi: context k encodes frames hcj_shard_range(n, k, nctx) on its own host thread.
int hcj_encode_batch_multi(hcj_ctx *const *ctx, int nctx, const uint8_t *const *yuv, int n, int width, int height, int chroma,
                           int quality, int restart_interval, uint8_t *const *out, const size_t *out_capacity, size_t *out_len,
                           int *status) {
  return hcj_encode_batch_multi_ex(ctx, nctx, yuv, n, width, height, chroma, quality, restart_interval, 0u, out, out_capacity,
                                   out_len, status);
}

int hcj_encode_batch_multi_ex(hcj_ctx *const *ctx, int nctx, const uint8_t *const *yuv, int n, int width, int height, int chroma,
                              int quality, int restart_interval, unsigned flags, uint8_t *const *out, const size_t *out_capacity,
                              size_t *out_len, int *status) {
  if (flags & ~HCJ_ENC_OPTIMIZE_HUFFMAN) return HCJ_ERR_INVALID_ARG;
  if (!ctx || nctx < 1 || n < 0 || (n > 0 && (!yuv || !out || !out_capacity || !out_len))) return HCJ_ERR_INVALID_ARG;
  for (int k = 0; k < nctx; k++) {
    if (!ctx[k]) return HCJ_ERR_INVALID_ARG;
    for (int j = 0; j < k; j++)
      if (ctx[k] == ctx[j]) return HCJ_ERR_INVALID_ARG;
  }
  std::vector<int> rc((size_t)nctx, HCJ_OK);
  auto work = [&](int k) {
    int lo, hi;
    hcj_shard_range(n, k, nctx, &lo, &hi);
    rc[k] = hcj_encode_batch_ex(ctx[k], yuv + lo, hi - lo, width, height, chroma, quality, restart_interval, flags, out + lo,
                                out_capacity + lo, out_len + lo, status ? status + lo : nullptr);
  };
  std::vector<std::thread> pool;
  try {
    for (int k = 1; k < nctx; k++) pool.emplace_back(work, k);
  } catch (...) {
    for (auto &t : pool) t.join();
    return HCJ_ERR_OUT_OF_MEMORY;
  }
  work(0);
  for (auto &t : pool) t.join();
  for (int k = 0; k < nctx; k++)
    if (rc[k] != HCJ_OK) return rc[k];
  return HCJ_OK;
}

int hcj_encode_last_device_ms(hcj_ctx *c, float *ms) {
  if (!c || !ms) return HCJ_ERR_INVALID_ARG;
  if (!c->enc_timed) return HCJ_ERR_INVALID_ARG;
  *ms = c->enc_ms;  // kernel time summed over the chunks of the call
  return HCJ_OK;
}

int hcj_encode_block_log(hcj_ctx *c, const uint8_t *yuv, int width, int height, int chroma, int quality, int restart_interval,
                         size_t first_block, size_t count, hcj_encoder_block *out) {
  static_assert(sizeof(hcj_encoder_block) == sizeof(hcjk::EncodeBlockLog), "hcj_encode_block_log layout");
  if (!c || !yuv || !out) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  EncodeSetup S;
  int st = setup_encode(c, 1, width, height, chroma, quality, restart_interval, false, &S);
  if (st == HCJ_OK && (first_block > S.dev.nblocks || count > S.dev.nblocks - first_block)) st = HCJ_ERR_INVALID_ARG;
  cudaError_t err = cudaSuccess;
  void *d_out = nullptr;
  if (st == HCJ_OK && count) st = c->alloc(&d_out, count * sizeof(hcj_encoder_block));
  if (st == HCJ_OK && count) {
    S.owned.push_back(d_out);
    hcjk::EncodeBatchDev &e = S.dev;
    err = cudaMemcpyAsync(const_cast<uint8_t *>(e.src), yuv, e.frame_bytes, cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess) {
      hcjk::launch_encode(e, c->stream);  // Block.quant of every block: the DC predictors
      hcjk::launch_encode_block_log(e, (uint32_t)first_block, (uint32_t)count, d_out, c->stream);
      err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaMemcpyAsync(out, d_out, count * sizeof(hcj_encoder_block), cudaMemcpyDeviceToHost, c->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
  }
  teardown_encode(c, &S);
  if (st != HCJ_OK) return st;
  return err == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)err;
}

int hcj_encode_quantized(hcj_ctx *c, const uint8_t *yuv, int width, int height, int chroma, int quality, int16_t *quant,
                         size_t capacity_blocks) {
  if (!c || !yuv || !quant) return HCJ_ERR_INVALID_ARG;
  CU_TRY(cudaSetDevice(c->device));
  EncodeSetup S;
  int st = setup_encode(c, 1, width, height, chroma, quality, 0, false, &S);
  if (st == HCJ_OK && capacity_blocks < S.dev.nblocks) st = HCJ_ERR_BUFFER_TOO_SMALL;
  cudaError_t err = cudaSuccess;
  if (st == HCJ_OK) {
    hcjk::EncodeBatchDev &e = S.dev;
    err = cudaMemcpyAsync(const_cast<uint8_t *>(e.src), yuv, e.frame_bytes, cudaMemcpyHostToDevice, c->stream);
    if (err == cudaSuccess) {
      hcjk::launch_encode(e, c->stream);
      err = cudaGetLastError();
    }
    if (err == cudaSuccess) err = cudaMemcpyAsync(quant, e.quant, (size_t)e.nblocks * 128, cudaMemcpyDeviceToHost, c->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(c->stream);
  }
  teardown_encode(c, &S);
  if (st != HCJ_OK) return st;
  return err == cudaSuccess ? HCJ_OK : HCJ_ERR_CUDA - (int)err;
}

}  // extern "C"
