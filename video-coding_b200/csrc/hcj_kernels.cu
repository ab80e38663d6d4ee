// hcj_kernels.cu — decode kernels for sm_100a.
//
//   k_destuff                          D3  extract_entropy_coded_bits (decoder.ml:261-281) + restart-marker scan in one
//                                          pass: a chained scan with decoupled look-back over 4 KiB tiles
//                                          (k_destuff_count / _scan / _write: the three-kernel form, HCJ_DESTUFF_3PASS)
//   k_huff_restart                     D6  huffman_decode per SHORT restart interval (stated extension), DC
//                                          resolved in-thread: fast steps in lock step per block
//   k_spec_units / _sync / _fix /      D6  huffman_decode of scans without restart markers and of LONG restart
//   _write                                 intervals: self-synchronising speculative subsequence decode over the whole
//                                          batch (one pass with a guessed-state warm-up, multi-symbol AC look-ups),
//                                          per-image fix-point on a compacted list, segmented prefix sums for block
//                                          indices and DC predictors (decoder.ml:118-165,347-397), exact pass on whole MCUs
//   k_idct_persistent                  D7-D11 dequantise + inverse zig-zag + Chen IDCT + clip/level-shift + crop + store;
//                                          the FUSED instance also converts to RGB24 inside the tile (4:4:4; sub-sampled
//                                          opt-in, k_rgb_deferred / k_rgb444_fix finish it)
//   k_rgb, k_rgb_sub_pairs             D12/D13 Planar_444 up-sampling + stated YCbCr->RGB from the plane buffer
//   k_idct_blocks, k_block_log, k_compare*  debug taps (Component.recon, Component.Summary), Ocompare on the device
//
// None of this is GEMM-shaped: no tensor cores.  The entropy kernels are bound by instruction issue and
// shared-memory table look-ups, the IDCT kernel by integer issue at 67 % of the HBM roofline (DESIGN.md has
// the byte counts and the ncu numbers).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "hcj_device.cuh"
#include "hcj_kernels.cuh"

namespace hcjk {

using namespace hcjdev;

// ================================================================================================
// K1: destuff + marker scan (extract_entropy_coded_bits, decoder.ml:261-281, + RSTn splitting).
// The scan of every image is cut into 4 KiB tiles; a byte's fate depends only on itself and its
// predecessor, exactly as in the model's recursive search_for_marker, so tiles are independent:
//   k_destuff_count  per tile: bytes kept, restart markers, position of the first terminating marker
//   k_destuff_scan   per image: the first tile with a terminator ends the scan; exclusive scan of the
//                    counts before it -> every tile's output offset and first interval index; image state
//   k_destuff_write  per tile: compacts its bytes (block scan), stages them in shared memory at the same
//                    16-byte phase as their destination and writes aligned 16-byte words (+ the partial
//                    words at both ends byte by byte); interval start offsets go to seg_offs
// All three run over (tile, image) grids, so one large image fills the GPU as well as many small ones.
// ================================================================================================
constexpr int DS_THREADS = 256;
constexpr uint32_t DS_TILE = DS_THREADS * 16;

__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, v, d);
    if (lane >= d) v += t;
  }
  return v;
}

// The 16 bytes of one thread classified, four bytes at a time: every mask below is a word with 0x80 in the
// bytes that have the property (SIMD within a register: no per-byte loop on the common path).
//   emit  the byte is kept (for an FF 00 pair: the 00 position keeps the deferred FF, see ffz)
//   mark  second byte of a restart marker        term  second byte of any other marker (ends the scan)
//   ffz   00 that follows FF: emits FF            ff    the byte is FF
struct DsClass {
  uint32_t w[4];
  uint32_t emit[4], mark[4], term[4], ffz[4];
  uint32_t anyff;  // some byte of the 16 is FF, or the byte before them is: the bytes are not kept verbatim
};
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {  // 0x80 in every byte of x that is 0 (exact)
  return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu);
}
__device__ __forceinline__ DsClass ds_classify(const uint8_t *file, uint32_t off, uint32_t start, uint32_t flen, bool restart) {
  DsClass c;
  uint4 v = make_uint4(0, 0, 0, 0);
  if (off < flen) v = __ldg(reinterpret_cast<const uint4 *>(file + off));
  // the byte in front of the 16: its own load (the line is the neighbour thread's, an L1 hit) instead of an exchange
  // through shared memory and a CTA barrier
  const uint32_t prev = (off > start && off - 1 < flen) ? (uint32_t)__ldg(file + off - 1) : 0u;
  c.w[0] = v.x, c.w[1] = v.y, c.w[2] = v.z, c.w[3] = v.w;
  // the model starts with prev = '\x00' (decoder.ml:279): the byte before `start` does not count
  uint32_t pff = (prev == 0xffu && off != start) ? 0x80u : 0u;  // "the previous byte is FF", for byte 0 of the word
  c.anyff = pff;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const uint32_t w = c.w[k];
    const uint32_t ff = zero_bytes(~w), zz = zero_bytes(w);
    const uint32_t rst = restart ? zero_bytes((w & 0xf8f8f8f8u) ^ 0xd0d0d0d0u) : 0u;
    const uint32_t p = (ff << 8) | pff;  // previous byte is FF
    c.ffz[k] = p & zz;
    c.emit[k] = (p & zz) | (~p & ~ff & 0x80808080u);
    c.mark[k] = p & rst;
    c.term[k] = p & ~zz & ~rst;
    c.anyff |= ff;
    pff = ff >> 24;
  }
  // bytes outside [start, flen) do not exist (first and last tile of the scan only)
  if (off < start || off + 16u > flen) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint32_t in = 0;
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const uint32_t pos = off + 4 * k + i;
        if (pos >= start && pos < flen) in |= 0x80u << (8 * i);
      }
      // a marker / stuffed pair straddling `start` cannot happen (prev is forced to 0 there); mask everything
      c.emit[k] &= in;
      c.mark[k] &= in;
      c.term[k] &= in;
      c.ffz[k] &= in;
    }
    c.anyff |= 0x80u;  // take the byte-wise path
    // the byte at `start` sees prev = 0 even if the byte before it is FF
    if (start > off && start < off + 16u) {
      const uint32_t k = (start - off) >> 2, i = (start - off) & 3u, bit = 0x80u << (8 * i);
      const uint32_t wk = k == 0 ? c.w[0] : k == 1 ? c.w[1] : k == 2 ? c.w[2] : c.w[3];  // (no run-time index: the words stay in registers)
      const uint32_t ch = (wk >> (8 * i)) & 0xffu;
#pragma unroll
      for (int kk = 0; kk < 4; kk++)
        if ((uint32_t)kk == k) {
          c.mark[kk] &= ~bit;
          c.term[kk] &= ~bit;
          c.ffz[kk] &= ~bit;
          c.emit[kk] = (c.emit[kk] & ~bit) | (ch != 0xffu ? bit : 0u);
        }
    }
  }
  return c;
}
__device__ __forceinline__ uint32_t ds_count(const uint32_t m[4]) {
  return (uint32_t)(__popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]));
}
// first terminator of the tile (block-wide min), 0xffffffff if none; drops everything at or after it
__device__ __forceinline__ uint32_t ds_cut_at_terminator(DsClass &c, uint32_t off, uint32_t *s_min, int lane, int warp) {
  uint32_t tpos = 0xffffffffu;
  // a terminating marker is in the last tile of a scan only: every other tile leaves after one barrier
  if (!__syncthreads_or((c.term[0] | c.term[1] | c.term[2] | c.term[3]) != 0u)) return tpos;
  if (c.term[0] | c.term[1] | c.term[2] | c.term[3]) {
#pragma unroll
    for (int k = 3; k >= 0; k--)
      if (c.term[k]) tpos = off + 4 * k + (((uint32_t)__ffs((int)c.term[k]) - 1u) >> 3);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) tpos = min(tpos, __shfl_xor_sync(0xffffffffu, tpos, s));
  if (lane == 0) s_min[warp] = tpos;
  __syncthreads();
  uint32_t tmin = s_min[0];
#pragma unroll
  for (int k = 1; k < DS_THREADS / 32; k++) tmin = min(tmin, s_min[k]);
  if (tmin != 0xffffffffu && off + 16 > tmin) {
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint32_t keep = 0;
#pragma unroll
      for (int i = 0; i < 4; i++)
        if (off + 4 * k + i < tmin) keep |= 0x80u << (8 * i);
      c.emit[k] &= keep;
      c.mark[k] &= keep;
      c.ffz[k] &= keep;
    }
    c.anyff |= 0x80u;
  }
  return tmin;
}

struct DsTile {
  uint32_t counts;  // after k_destuff_count: kept bytes | markers << 16; after k_destuff_scan: output offset (0xffffffff = dropped)
  uint32_t term;    // after k_destuff_count: first terminator or 0xffffffff; after k_destuff_scan: first interval index
};

__device__ __forceinline__ bool ds_tile_setup(const DecodeBatchDev &b, const HcjImageDesc *&d, uint32_t &off) {
  d = &b.descs[blockIdx.y + b.img_lo];
  if (!d->valid) return false;
  const uint32_t base0 = d->scan_start & ~15u;
  if (base0 + (uint64_t)blockIdx.x * DS_TILE >= d->file_len) return false;
  off = base0 + blockIdx.x * DS_TILE + threadIdx.x * 16;
  return true;
}

__global__ void __launch_bounds__(DS_THREADS) k_destuff_count(DecodeBatchDev b) {
  __shared__ uint32_t s_min[DS_THREADS / 32];
  __shared__ uint32_t s_cnt[DS_THREADS / 32];
  const HcjImageDesc *d;
  uint32_t off;
  if (!ds_tile_setup(b, d, off)) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  DsClass c = ds_classify(b.files + d->file_off, off, d->scan_start, d->file_len, d->ri > 0);
  const uint32_t tmin = ds_cut_at_terminator(c, off, s_min, lane, warp);
  uint32_t cnt = (ds_count(c.mark) << 16) | ds_count(c.emit);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, s);
  if (lane == 0) s_cnt[warp] = cnt;
  __syncthreads();
  if (tid == 0) {
    uint32_t total = 0;
#pragma unroll
    for (int k = 0; k < DS_THREADS / 32; k++) total += s_cnt[k];
    DsTile t;
    t.counts = total;
    t.term = tmin;
    b.ds_tiles[d->ds_off + blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(DS_THREADS) k_destuff_scan(DecodeBatchDev b) {
  __shared__ uint32_t s_warp[DS_THREADS / 32];
  __shared__ uint32_t s_first;
  const int img = blockIdx.x + b.img_lo;
  const HcjImageDesc &d = b.descs[img];
  if (!d.valid) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t base0 = d.scan_start & ~15u;
  const uint32_t ntiles = d.file_len > base0 ? (d.file_len - base0 + DS_TILE - 1) / DS_TILE : 0;
  DsTile *tiles = b.ds_tiles + d.ds_off;
  // the first tile that holds a terminator ends the scan
  if (tid == 0) s_first = 0xffffffffu;
  __syncthreads();
  for (uint32_t t0 = 0; t0 < ntiles; t0 += DS_THREADS) {
    const uint32_t t = t0 + tid;
    const bool has = t < ntiles && tiles[t].term != 0xffffffffu;
    const uint32_t m = __ballot_sync(0xffffffffu, has);
    if (m && lane == 0) atomicMin(&s_first, t0 + warp * 32 + (uint32_t)__ffs((int)m) - 1u);
    __syncthreads();
    if (s_first != 0xffffffffu) break;
  }
  const uint32_t first = s_first;
  const bool found = first != 0xffffffffu;
  const uint32_t nlive = found ? first + 1 : ntiles;
  uint32_t carry = 0;  // kept bytes | markers << 16 (a scan has far fewer than 2^16 restart intervals... checked on the host)
  uint32_t carry_mark = 0;
  for (uint32_t t0 = 0; t0 < ntiles; t0 += DS_THREADS) {
    const uint32_t t = t0 + tid;
    const uint32_t v = t < nlive ? tiles[t].counts : 0u;
    const uint32_t ve = v & 0xffffu, vm = v >> 16;
    // two scans in one: bytes in the low half would overflow 16 bits, so scan them separately
    uint32_t ie = warp_incl_scan(ve, lane), im = warp_incl_scan(vm, lane);
    __syncthreads();
    if (lane == 31) s_warp[warp] = ie;
    __syncthreads();
    uint32_t be = 0, te = 0;
#pragma unroll
    for (int k = 0; k < DS_THREADS / 32; k++) {
      const uint32_t x = s_warp[k];
      if (k < warp) be += x;
      te += x;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = im;
    __syncthreads();
    uint32_t bm = 0, tm = 0;
#pragma unroll
    for (int k = 0; k < DS_THREADS / 32; k++) {
      const uint32_t x = s_warp[k];
      if (k < warp) bm += x;
      tm += x;
    }
    if (t < ntiles) {
      DsTile o;
      o.counts = t < nlive ? carry + be + ie - ve : 0xffffffffu;
      o.term = carry_mark + bm + im - vm;
      tiles[t] = o;
    }
    carry += te;
    carry_mark += tm;
  }
  if (tid == 0) {
    uint32_t *segs = b.seg_offs + d.seg_off;
    HcjImageState st;
    st.ent_len = carry;
    st.nseg_found = carry_mark + 1;
    st.status = HCJ_DEV_OK;
    st.pad_ = 0;
    st.err_key = HCJ_NO_ERR_KEY;
    if (!found) st.status = HCJ_DEV_NO_TERMINATOR;
    else if (d.ri > 0 && st.nseg_found != d.nseg_expected) st.status = HCJ_DEV_RESTART_COUNT;
    segs[0] = 0;
    segs[d.nseg_expected] = carry;
    b.states[img] = st;
  }
}

__global__ void __launch_bounds__(DS_THREADS) k_destuff_write(DecodeBatchDev b) {
  __shared__ uint32_t s_warp[DS_THREADS / 32];
  __shared__ uint32_t s_min[DS_THREADS / 32];
  // Compacted bytes of the tile, placed at the same 16-byte phase as their destination.  Zeroed first:
  // a thread ORs the words it shares with its neighbours and stores the ones that are wholly its own.
  __shared__ __align__(16) uint32_t s_out[(DS_TILE + 32) / 4];
  const HcjImageDesc *d;
  uint32_t off;
  if (!ds_tile_setup(b, d, off)) return;
  const DsTile tile = b.ds_tiles[d->ds_off + blockIdx.x];
  if (tile.counts == 0xffffffffu) return;  // behind the terminator
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  reinterpret_cast<uint4 *>(s_out)[tid] = make_uint4(0u, 0u, 0u, 0u);
  if (tid < 2) reinterpret_cast<uint4 *>(s_out)[DS_THREADS + tid] = make_uint4(0u, 0u, 0u, 0u);
  uint8_t *ent = b.entropy + d->ent_off;
  uint32_t *segs = b.seg_offs + d->seg_off;
  const uint32_t nseg_expected = d->nseg_expected;
  DsClass c = ds_classify(b.files + d->file_off, off, d->scan_start, d->file_len, d->ri > 0);
  ds_cut_at_terminator(c, off, s_min, lane, warp);
  // block exclusive scan of (markers << 16 | kept bytes): at most 4096 bytes and 2048 markers per tile
  const uint32_t cnt = (ds_count(c.mark) << 16) | ds_count(c.emit);
  const uint32_t incl = warp_incl_scan(cnt, lane);
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();  // also orders the zeroing of s_out before the ORs below
  uint32_t wbase = 0, total = 0;
#pragma unroll
  for (int k = 0; k < DS_THREADS / 32; k++) {
    const uint32_t t = s_warp[k];
    if (k < warp) wbase += t;
    total += t;
  }
  const uint32_t excl = wbase + incl - cnt;
  const uint32_t out0 = tile.counts, phase = out0 & 15u;
  const uint32_t so = phase + (excl & 0xffffu);
  if (c.anyff == 0u) {
    // all 16 bytes kept verbatim: shift them to the byte phase of their place and store word-wise
    const uint32_t q = so >> 2, sh = (so & 3u) * 8u;
    if (sh == 0u) {
      s_out[q] = c.w[0], s_out[q + 1] = c.w[1], s_out[q + 2] = c.w[2], s_out[q + 3] = c.w[3];
    } else {
      atomicOr(&s_out[q], c.w[0] << sh);
      s_out[q + 1] = __funnelshift_l(c.w[0], c.w[1], sh);
      s_out[q + 2] = __funnelshift_l(c.w[1], c.w[2], sh);
      s_out[q + 3] = __funnelshift_l(c.w[2], c.w[3], sh);
      atomicOr(&s_out[q + 4], c.w[3] >> (32u - sh));
    }
  } else {
    // some byte of the 16 is special: words that are still kept verbatim go as a unit, the others byte by byte
    uint32_t o = so, opos = out0 + (excl & 0xffffu), mk = tile.term + (excl >> 16);
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (c.emit[k] == 0x80808080u && c.ffz[k] == 0u) {
        const uint32_t sh = (o & 3u) * 8u;
        if (sh == 0u) {
          s_out[o >> 2] = c.w[k];
        } else {
          atomicOr(&s_out[o >> 2], c.w[k] << sh);
          atomicOr(&s_out[(o >> 2) + 1], c.w[k] >> (32u - sh));
        }
        o += 4;
        opos += 4;
      } else if ((c.emit[k] | c.mark[k]) != 0u) {
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const uint32_t bit = 0x80u << (8 * i);
          if (c.emit[k] & bit) {
            const uint32_t ch = (c.ffz[k] & bit) ? 0xffu : (c.w[k] >> (8 * i)) & 0xffu;
            atomicOr(&s_out[o >> 2], ch << ((o & 3u) * 8u));
            o++;
            opos++;
          } else if (c.mark[k] & bit) {
            mk++;
            if (mk < nseg_expected) segs[mk] = opos;  // interval mk starts here
          }
        }
      }
    }
  }
  __syncthreads();
  const uint8_t *s_bytes = reinterpret_cast<const uint8_t *>(s_out);
  const uint32_t nbytes = total & 0xffffu, avail = phase + nbytes;
  uint8_t *dst0 = ent + (out0 - phase);  // 16-byte aligned
  const uint32_t w_lo = phase ? 1u : 0u, w_hi = avail >> 4;  // words [w_lo, w_hi) are wholly this tile's
  for (uint32_t k = w_lo + tid; k < w_hi; k += DS_THREADS)
    reinterpret_cast<uint4 *>(dst0)[k] = reinterpret_cast<const uint4 *>(s_out)[k];
  // partial words at both ends (shared with the neighbouring tiles): byte by byte
  if (phase && (uint32_t)tid < 16u - phase && phase + tid < avail) dst0[phase + tid] = s_bytes[phase + tid];
  const uint32_t tail0 = max(w_hi << 4, w_lo << 4);
  if (tail0 + tid < avail && tail0 + tid >= phase && (uint32_t)tid < 16u) dst0[tail0 + tid] = s_bytes[tail0 + tid];
}

// ------------------------------------------------------------------------------------------------
// The same in ONE pass (the input is read once): every tile classifies its bytes, scans them, and learns what
// lies before it from the records of its predecessors - a chained scan with decoupled look-back (Merrill & Garland)
// over the tiles of an image.  A tile's record is one 64-bit word, so status and value are published by a
// single store:
//   bits 0-31 kept bytes | bits 32-59 restart markers | bit 60 a terminating marker was seen | bits 62-63 status
//   status 0 = not yet written (the records are zeroed before every decode), 1 = this tile alone, 2 = this tile
//   and everything before it.
// Tiles are looked at by warp 0, 32 predecessors per step.  A tile only ever waits for tiles with a smaller block
// index of the same image row of the grid, which the hardware has dispatched before it.
// ------------------------------------------------------------------------------------------------
constexpr unsigned long long DSR_VALUE = (1ull << 60) - 1ull, DSR_TERM = 1ull << 60;
__device__ __forceinline__ unsigned long long dsr_load(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void dsr_store(unsigned long long *p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__device__ __forceinline__ void ds_write_state(const DecodeBatchDev &b, const HcjImageDesc *d, uint32_t img, uint32_t ent_len,
                                               uint32_t markers, bool found) {
  uint32_t *segs = b.seg_offs + d->seg_off;
  HcjImageState st;
  st.ent_len = ent_len;
  st.nseg_found = markers + 1;
  st.status = HCJ_DEV_OK;
  st.pad_ = 0;
  st.err_key = HCJ_NO_ERR_KEY;
  if (!found) st.status = HCJ_DEV_NO_TERMINATOR;
  else if (d->ri > 0 && st.nseg_found != d->nseg_expected) st.status = HCJ_DEV_RESTART_COUNT;
  segs[0] = 0;
  segs[d->nseg_expected] = ent_len;
  b.states[img] = st;
}

__global__ void __launch_bounds__(DS_THREADS) k_destuff(DecodeBatchDev b) {
  __shared__ uint32_t s_warp[DS_THREADS / 32];
  __shared__ uint32_t s_min[DS_THREADS / 32];
  __shared__ unsigned long long s_prefix;
  __shared__ __align__(16) uint32_t s_out[(DS_TILE + 32) / 4];  // the tile's kept bytes, compacted from offset 0
  __shared__ uint32_t s_sel[16];  // byte-permute selector that squeezes a word's kept bytes (flags = index) to its low end
  if (threadIdx.x < 16) {
    uint32_t sel = 0x4444u, n = 0;  // 4 = a byte of the zero operand
    for (uint32_t i = 0; i < 4; i++)
      if (threadIdx.x >> i & 1u) {
        sel = (sel & ~(0xfu << (4 * n))) | (i << (4 * n));
        n++;
      }
    s_sel[threadIdx.x] = sel;  // published by the barrier inside ds_cut_at_terminator
  }
  // grid (images, tiles): CTAs are dispatched image-fastest, so the tiles in flight at any moment are about the same
  // tile of many images and a tile's predecessors have long published their inclusive records (tile-fastest, all tiles
  // of one large image start together and every look-back walks back through hundreds of records: 2.08 ms against
  // 1.94 ms for the three kernels on 128 x 4k 4:4:4)
  const uint32_t img = blockIdx.x + b.img_lo;
  const HcjImageDesc *d = &b.descs[img];
  if (!d->valid) return;
  const uint32_t base0 = d->scan_start & ~15u;
  const uint32_t ntiles = d->file_len > base0 ? (d->file_len - base0 + DS_TILE - 1) / DS_TILE : 0;
  const uint32_t t = blockIdx.y;
  if (t >= ntiles) {
    if (t == 0 && threadIdx.x == 0) ds_write_state(b, d, img, 0, 0, false);  // a scan of zero bytes has no terminator
    return;
  }
  const uint32_t off = base0 + t * DS_TILE + threadIdx.x * 16;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  reinterpret_cast<uint4 *>(s_out)[tid] = make_uint4(0u, 0u, 0u, 0u);
  if (tid < 2) reinterpret_cast<uint4 *>(s_out)[DS_THREADS + tid] = make_uint4(0u, 0u, 0u, 0u);
  DsClass c = ds_classify(b.files + d->file_off, off, d->scan_start, d->file_len, d->ri > 0);
  const uint32_t tmin = ds_cut_at_terminator(c, off, s_min, lane, warp);
  // block exclusive scan of (markers << 16 | kept bytes): at most 4096 bytes and 2048 markers per tile
  const uint32_t cnt = (ds_count(c.mark) << 16) | ds_count(c.emit);
  const uint32_t incl = warp_incl_scan(cnt, lane);
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();  // also orders the zeroing of s_out before the ORs below
  uint32_t wbase = 0, total = 0;
#pragma unroll
  for (int k = 0; k < DS_THREADS / 32; k++) {
    const uint32_t x = s_warp[k];
    if (k < warp) wbase += x;
    total += x;
  }
  const uint32_t excl = wbase + incl - cnt;
  // ---- publish this tile's own counts at once: the tiles behind it can look back while this one compacts
  unsigned long long *recs = reinterpret_cast<unsigned long long *>(b.ds_tiles + d->ds_off);
  const unsigned long long mine = (unsigned long long)(total & 0xffffu) | ((unsigned long long)(total >> 16) << 32) |
                                  (tmin != 0xffffffffu ? DSR_TERM : 0ull);
  if (tid == 0) dsr_store(recs + t, mine | ((t == 0 ? 2ull : 1ull) << 62));
  // ---- compact the tile's kept bytes into shared memory, from offset 0
  const uint32_t so = excl & 0xffffu;
  if (c.anyff == 0u) {
    const uint32_t q = so >> 2, sh = (so & 3u) * 8u;
    if (sh == 0u) {
      s_out[q] = c.w[0], s_out[q + 1] = c.w[1], s_out[q + 2] = c.w[2], s_out[q + 3] = c.w[3];
    } else {
      atomicOr(&s_out[q], c.w[0] << sh);
      s_out[q + 1] = __funnelshift_l(c.w[0], c.w[1], sh);
      s_out[q + 2] = __funnelshift_l(c.w[1], c.w[2], sh);
      s_out[q + 3] = __funnelshift_l(c.w[2], c.w[3], sh);
      atomicOr(&s_out[q + 4], c.w[3] >> (32u - sh));
    }
  } else {
    // some byte goes (or an FF arrives late, behind its 00): every word is squeezed by ONE byte permute whose selector
    // comes from a 16-entry table indexed by the word's four keep flags, and ORed in at its byte offset.  No branches:
    // the few lanes of a warp that are here (6 % of the threads, but some lane of 86 % of the warps) run in step,
    // whatever word their FF sits in (the byte loop this replaces ran its four cases one after the other).
    uint32_t o = so;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const uint32_t e = c.emit[k];
      const uint32_t w2 = c.w[k] | ((c.ffz[k] >> 7) * 0xffu);                  // the 00 behind an FF emits the FF
      const uint32_t sel = s_sel[((e >> 7) * 0x10204080u) >> 28];              // flags of bytes 0..3 -> bits 0..3
      const uint32_t v = __byte_perm(w2, 0u, sel);                             // kept bytes at the low end, zeros above
      const uint32_t sh = (o & 3u) * 8u;
      atomicOr(&s_out[o >> 2], v << sh);
      atomicOr(&s_out[(o >> 2) + 1], __funnelshift_l(v, 0u, sh));              // v >> (32 - sh); 0 for sh = 0
      o += (uint32_t)__popc(e);
    }
  }
  // ---- what lies before this tile (warp 0; by now the predecessors have mostly published)
  if (warp == 0) {
    unsigned long long before = 0;  // value and terminator bit of everything before this tile
    if (t != 0) {
      int base = (int)t - 1;
      for (;;) {
        const int idx = base - lane;
        unsigned long long v = 2ull << 62;  // before tile 0: nothing, and final
        if (idx >= 0) {
          v = dsr_load(recs + idx);
          while ((v >> 62) == 0ull) v = dsr_load(recs + idx);
        }
        const uint32_t final_mask = __ballot_sync(0xffffffffu, (v >> 62) == 2ull);
        const int first = final_mask ? __ffs((int)final_mask) - 1 : 31;  // lanes up to the nearest final record count
        unsigned long long part = lane <= first ? (v & DSR_VALUE) : 0ull;
        const uint32_t term_mask = __ballot_sync(0xffffffffu, lane <= first && (v & DSR_TERM) != 0ull);
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) part += __shfl_xor_sync(0xffffffffu, part, sft);
        before += part;
        if (term_mask) before |= DSR_TERM;
        if (final_mask) break;
        base -= 32;
      }
      if (lane == 0) dsr_store(recs + t, ((before & DSR_VALUE) + (mine & DSR_VALUE)) | ((before | mine) & DSR_TERM) | (2ull << 62));
    }
    if (lane == 0) s_prefix = before;
  }
  __syncthreads();
  const unsigned long long before = s_prefix;
  if (before & DSR_TERM) return;  // behind the terminator: the model never looks at these bytes
  const uint32_t out0 = (uint32_t)before, mk0 = (uint32_t)((before & DSR_VALUE) >> 32);
  if (tid == 0 && (tmin != 0xffffffffu || t + 1 == ntiles))
    ds_write_state(b, d, img, out0 + (total & 0xffffu), mk0 + (total >> 16), tmin != 0xffffffffu);
  // ---- restart markers: interval mk starts at the output position of the byte behind the marker
  if (c.mark[0] | c.mark[1] | c.mark[2] | c.mark[3]) {
    uint32_t *segs = b.seg_offs + d->seg_off;
    const uint32_t nseg_expected = d->nseg_expected;
    uint32_t opos = out0 + (excl & 0xffffu), mk = mk0 + (excl >> 16);
    // one iteration per marker (a lane rarely holds more than one), not one per byte: the interval starts at the
    // output position of the bytes kept in front of the marker
#pragma unroll
    for (int k = 0; k < 4; k++) {
      uint32_t m = c.mark[k] & ~c.emit[k];  // (a flag is never both; the byte loop this replaces gave emit precedence)
      while (m) {
        const uint32_t bit = m & (0u - m);  // the lowest flag = the first marker of the word
        mk++;
        if (mk < nseg_expected) segs[mk] = opos + (uint32_t)__popc(c.emit[k] & (bit - 1u));
        m ^= bit;
      }
      opos += (uint32_t)__popc(c.emit[k]);
    }
  }
  // ---- copy out: destination word k (16 bytes, aligned) takes the tile's bytes [16 k - phase, 16 k - phase + 16)
  uint8_t *ent = b.entropy + d->ent_off;
  const uint32_t phase = out0 & 15u, nbytes = total & 0xffffu, avail = phase + nbytes;
  uint8_t *dst0 = ent + (out0 - phase);  // 16-byte aligned
  const uint8_t *s_bytes = reinterpret_cast<const uint8_t *>(s_out);
  const uint32_t w_lo = phase ? 1u : 0u, w_hi = avail >> 4;  // words [w_lo, w_hi) are wholly this tile's
  for (uint32_t k = w_lo + tid; k < w_hi; k += DS_THREADS) {
    const uint32_t sb = 16u * k - phase;  // first source byte
    const uint32_t q = sb >> 2, sh = (sb & 3u) * 8u;
    const uint32_t a0 = s_out[q], a1 = s_out[q + 1], a2 = s_out[q + 2], a3 = s_out[q + 3], a4 = s_out[q + 4];
    reinterpret_cast<uint4 *>(dst0)[k] = make_uint4(__funnelshift_r(a0, a1, sh), __funnelshift_r(a1, a2, sh), __funnelshift_r(a2, a3, sh),
                                                    __funnelshift_r(a3, a4, sh));
  }
  // partial words at both ends (shared with the neighbouring tiles): byte by byte
  if (phase && (uint32_t)tid < 16u - phase && (uint32_t)tid < nbytes) dst0[phase + tid] = s_bytes[tid];
  const uint32_t tail0 = max(w_hi << 4, w_lo << 4);
  if (tail0 + tid < avail && tail0 + tid >= phase && (uint32_t)tid < 16u) dst0[tail0 + tid] = s_bytes[tail0 + tid - phase];
}

static bool destuff_three_pass() {
  // Measured on a B200 (profiles/r02_experiments/r02x_*, 1024 x 1080p / 128 x 4k 4:4:4 q95): three kernels 0.886 / 1.94 ms; the chained
  // scan with the look-back in front of the compaction and a tile-fastest grid 1.07 / 2.89 ms; with every tile's own
  // counts published before it compacts, the look-back behind the compaction and an image-fastest grid 0.74 / 1.58 ms.
  // HCJ_DESTUFF_3PASS=1 selects the three kernels (A/B measurements, tests).
  return getenv("HCJ_DESTUFF_3PASS") != nullptr;
}

void launch_destuff(const DecodeBatchDev &b, cudaStream_t s) {
  if (!destuff_three_pass() && b.max_ds_tiles <= 65535u) {  // (tiles are the grid's y dimension)
    if (b.img_hi <= b.img_lo) return;
    k_destuff<<<dim3(b.img_hi - b.img_lo, b.max_ds_tiles ? b.max_ds_tiles : 1u), DS_THREADS, 0, s>>>(b);
    return;
  }
  if (b.img_hi <= b.img_lo) return;
  // the per-image scan always runs: it writes the image state (a scan of zero bytes has no terminator)
  const dim3 grid(b.max_ds_tiles, b.img_hi - b.img_lo);
  if (b.max_ds_tiles) k_destuff_count<<<grid, DS_THREADS, 0, s>>>(b);
  k_destuff_scan<<<b.img_hi - b.img_lo, DS_THREADS, 0, s>>>(b);
  if (b.max_ds_tiles) k_destuff_write<<<grid, DS_THREADS, 0, s>>>(b);
}
int decode_prologue(const DecodeBatchDev &b, cudaStream_t s) {
  // Coefficient blocks are cleared (clear_block, decoder.ml:112-116,160) by the entropy kernels themselves, block by
  // block, right before they store into them (see zero_block in hcj_device.cuh).
  cudaError_t e = cudaMemsetAsync(b.wide_flags, 0, (size_t)(b.total_blocks / 32 + 2) * 4, s);
  if (e == cudaSuccess) e = cudaMemsetAsync(b.states, 0xff, sizeof(HcjImageState) * (size_t)b.n, s);  // overwritten by k_destuff for valid images
  if (e == cudaSuccess) e = cudaMemsetAsync(b.ds_tiles, 0, sizeof(DsTile) * ((size_t)b.total_ds_tiles + 1), s);
  return (int)e;
}
int destuff_kernel_count() { return destuff_three_pass() ? 3 : 1; }

// ================================================================================================
// Huffman tables in shared memory, shared by K2 and K3: per table HCJ_LUT_SIZE fast entries (32 bit,
// converted here from the host-built 16-bit primary table) + the second-level sub-tables.
// ================================================================================================
struct SmemTables {
  uint32_t max_bits[HCJ_MAX_COMP * 2];
  const uint16_t *full[HCJ_MAX_COMP * 2];
  uint8_t comp_pair[HCJ_MAX_COMP];
  uint8_t blk_comp[HCJ_MAX_BPM + 2];
  BlkInfo blkinfo[HCJ_MAX_BPM + 2];
  int32_t quant[HCJ_MAX_COMP * 128];  // per scan component: 64 plain entries + 64 in dp2a form
};
constexpr int LUT_SUB_ENTRIES = HCJ_LUT_NSUB * HCJ_LUT_SUB_SIZE;

// Bytes of shared memory behind a kernel's other dynamic shared memory: fast entries, then sub-tables.
static inline size_t lut_smem_bytes(const DecodeBatchDev &b) {
  return (size_t)b.max_pairs * 2 * (HCJ_LUT_SIZE + LUT_SUB_ENTRIES) * sizeof(uint32_t);
}

__device__ __forceinline__ FastTables load_tables(SmemTables &st, void *lut_smem, const DecodeBatchDev &b, const HcjImageDesc &d) {
  const HcjTableSet &ts = b.table_sets[d.table_set];
  uint32_t *fast = reinterpret_cast<uint32_t *>(lut_smem);
  uint32_t *sub = fast + (size_t)b.max_pairs * 2 * HCJ_LUT_SIZE;
  const uint16_t *src = b.lut_primary + ts.primary_off;
  const uint32_t ntab = ts.npairs * 2;
  for (uint32_t i = threadIdx.x; i < ntab * HCJ_LUT_SIZE; i += blockDim.x) {
    const uint32_t ti = i >> HCJ_LUT_BITS, k = i & (HCJ_LUT_SIZE - 1);
    fast[i] = fast_entry_from_primary(__ldg(src + ti * HCJ_LUT_ENTRIES + k), ts.meta[ti >> 1][ti & 1].max_bits, (ti & 1u) == 0u);
  }
  for (uint32_t i = threadIdx.x; i < ntab * LUT_SUB_ENTRIES; i += blockDim.x) {
    const uint32_t ti = i / LUT_SUB_ENTRIES, k = i - ti * LUT_SUB_ENTRIES;
    // uniform shape: every sub-table indexed by the HCJ_LUT_SUB_BITS bits behind the primary index (sub_source_index)
    const uint32_t ks = (k & ~(uint32_t)(HCJ_LUT_SUB_SIZE - 1)) | sub_source_index(k & (HCJ_LUT_SUB_SIZE - 1), ts.meta[ti >> 1][ti & 1].max_bits);
    sub[i] = fast_entry_or_none(__ldg(src + ti * HCJ_LUT_ENTRIES + HCJ_LUT_SIZE + ks), (ti & 1u) == 0u);
  }
  if (threadIdx.x < HCJ_MAX_COMP * 2) {
    const HcjTableMeta &m = ts.meta[threadIdx.x >> 1][threadIdx.x & 1];
    st.max_bits[threadIdx.x] = m.max_bits;
    st.full[threadIdx.x] = b.lut_full + m.full_off;
  }
  if (threadIdx.x < HCJ_MAX_COMP) st.comp_pair[threadIdx.x] = (uint8_t)d.comp[threadIdx.x].pair;
  if (threadIdx.x < HCJ_MAX_BPM) {
    const uint32_t comp = d.blk_comp[threadIdx.x], pr = (uint32_t)d.comp[comp < HCJ_MAX_COMP ? comp : 0].pair;
    st.blk_comp[threadIdx.x] = (uint8_t)comp;
    uint32_t qmax = 0;
    if (threadIdx.x < (uint32_t)d.bpm)
      for (int e = 1; e < 64; e++) qmax = max(qmax, (uint32_t)__ldg(b.qtables + d.qt_off + comp * 128u + e));
    BlkInfo bi;
    bi.tdc = (pr * 2 + 0) * HCJ_LUT_SIZE;
    bi.tac = (pr * 2 + 1) * HCJ_LUT_SIZE;
    bi.qoff = comp * 128u;
    bi.comp_qmax = comp | (qmax << 8);
    st.blkinfo[threadIdx.x] = bi;
  }
  for (uint32_t i = threadIdx.x; i < (uint32_t)d.ncomp * 128; i += blockDim.x) st.quant[i] = __ldg(b.qtables + d.qt_off + i);
  FastTables T;
  T.fast = fast;
  T.sub = sub;
  T.max_bits = st.max_bits;
  T.full = st.full;
  T.blkinfo = st.blkinfo;
  T.quant = st.quant;
  return T;
}

__device__ __forceinline__ Tables tables_of(const SmemTables &st, uint32_t comp) {
  uint32_t pr = st.comp_pair[comp];
  Tables t;
  t.dc_off = (pr * 2 + 0) * HCJ_LUT_SIZE;
  t.ac_off = (pr * 2 + 1) * HCJ_LUT_SIZE;
  t.dc_max_bits = st.max_bits[pr * 2 + 0];
  t.ac_max_bits = st.max_bits[pr * 2 + 1];
  return t;
}

__device__ __forceinline__ void fill_scan_ctx(ScanCtx &sc, const SmemTables &st, const DecodeBatchDev &b,
                                              const HcjImageDesc &d, uint32_t total_bits) {
  if (threadIdx.x == 0) {
    sc.words = reinterpret_cast<const uint32_t *>(b.entropy + d.ent_off);
    sc.total_bits = total_bits;
    sc.bpm = d.bpm;
    sc.wide_flags = b.wide_flags;
    sc.blk_base = d.coef_off;
  }
  if (threadIdx.x < (uint32_t)d.ncomp) sc.tab[threadIdx.x] = tables_of(st, threadIdx.x);
}

__device__ __forceinline__ void raise_status(HcjImageState *st, int code, uint32_t bit_pos) {
  atomicMin(&st->err_key, ((unsigned long long)bit_pos << 8) | (unsigned long long)(-code));
}

// ================================================================================================
// K2: one thread per restart interval.  Intervals are byte aligned and start with every DC predictor
// at 0, so a thread owns its MCUs outright and writes resolved coefficients straight to HBM.
// ================================================================================================
constexpr int HR_ROW_WORDS = 36;  // a lane's staged block: 32 words + pad to 144 bytes (16-byte aligned rows, conflict-free 16-byte reads)
constexpr int HR_STAGE_WORDS = 32 * HR_ROW_WORDS;  // per warp

// ------------------------------------------------------------------------------------------------
// Warp-synchronous exact pass (the symbol semantics of subseq_write), shared by K2 and K3.
//
// Every lane decodes its own run of WHOLE MCUs: from an MCU boundary at bit position p it decodes the MCUs (blocks <
// nblocks_end) that begin before `hi` or at / beyond the end of the data (subseq_write).  All lanes of a warp are
// therefore in the same block-in-MCU at every step: luma blocks run in lock step with luma blocks.  The block in progress is staged in the lane's row of
// `stage` (shared memory, 36-word stride) and, once complete, written out by the warp as one 128-byte line:
// scattered 2-byte stores cost one L2 partial-sector transaction per symbol and were the bottleneck of the entropy
// kernels.  (K3's threads used to start mid-block at their subsequence boundary and share that block with their left
// neighbour: the shared blocks needed clearing in advance and 2-byte stores from both sides.  Now the synchronisation
// pass records where the first block of every subsequence begins, and the left neighbour finishes its last block.)
// ------------------------------------------------------------------------------------------------
struct PassIn {
  uint32_t p, cz, hi, end_bits;
  int32_t blk;          // index of the block in progress (at a block boundary: the previous one)
  int32_t pred[HCJ_MAX_COMP];
  int32_t nblocks_end;  // blocks >= this are not decoded
  uint32_t share;       // sum(|dequantised coefficient|) of the block in progress so far (wide-block guard)
  bool valid;
};

// Finished blocks staged in the rows of the lanes in `mask`: the warp writes them out four at a time, a
// quarter-warp per block (8 lanes x 16 bytes = the 128-byte line), and zeroes the rows.  Per block that is
// one shared-memory load, one shared-memory store and one global store wavefront, the same as a fully
// coalesced copy, for a fraction of the instructions of a block-at-a-time loop.
__device__ __forceinline__ void warp_store_full(uint32_t mask, int32_t blk, uint32_t *stage, int lane, int16_t *coefs) {
  const int quarter = lane >> 3, sub = lane & 7;
#pragma unroll
  for (int p = 0; p < 8; p++) {
    if (((mask >> (4 * p)) & 0xfu) == 0u) continue;  // warp-uniform
    const int l = 4 * p + quarter;
    const int32_t bidx = __shfl_sync(0xffffffffu, blk, l);
    if ((mask >> l) & 1u) {
      uint4 *src = reinterpret_cast<uint4 *>(stage + l * HR_ROW_WORDS) + sub;
      const uint4 v = *src;
      *src = make_uint4(0u, 0u, 0u, 0u);
      reinterpret_cast<uint4 *>(coefs + (size_t)bidx * 64)[sub] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Fast exact pass: the straight-line steps of hcj_device.cuh, warp-synchronous.  Lanes in the middle of
// a block decode AC symbols; lanes at a block boundary wait until every lane is there; then, in one go,
// the warp writes the finished blocks out (warp_store_full), and every lane moves to its next
// block-in-MCU and decodes its DC symbol.  Batching the per-block work keeps it out of the per-symbol
// instruction stream and runs it with all lanes active.  On return `in`
// holds the state of every lane at the point where it left (end of its range, 32 bits before the end of
// its data, or the symbol the literal loop has to look at); warp_exact_pass carries on from there.
// Returns HCJ_DEV_COEF_INDEX (and the position) for a lane whose run went past coefficient 63.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int warp_exact_fast(const ScanCtx &sc, const FastTables T, uint32_t *stage, int lane, PassIn &in,
                                               int16_t *coefs, uint32_t *err_pos) {
  const uint32_t bpm = sc.bpm;
  int16_t *row = reinterpret_cast<int16_t *>(stage + lane * HR_ROW_WORDS);
  const uint32_t lim = in.end_bits >= 32u ? in.end_bits - 32u : 0u;  // the unmasked reader is valid below this
  ExactLane s;
  s.c = in.cz >> 8;
  s.z = in.cz & 0xffu;
  s.blk = in.blk;
  s.p0 = in.pred[0], s.p1 = in.pred[1], s.p2 = in.pred[2], s.p3 = in.pred[3];
  s.share = in.share;
  s.sumabs = 0u;
  const bool entered = in.valid && in.p < lim;
  s.br.init(sc.words, entered ? in.p : 0u);
  exact_bind_block(s, T);
  int st = !entered ? 2 : s.z != 0u ? 0 : 1;   // 0 = mid-block, 1 = at a block boundary, 2 = left, 3 = left with an error
  int err = HCJ_DEV_OK;

  for (;;) {
    // every lane that is mid-block decodes AC symbols until its block ends; the warp moves on when the last
    // one is there.  (Serving boundary lanes earlier, in smaller groups, costs more instructions in the
    // per-block code than the waiting costs here: measured.)
    while (__any_sync(0xffffffffu, st == 0)) {
#pragma unroll
      for (int u = 0; u < 2; u++) {
        if (st == 0) {
          if (s.br.pos >= lim) {
            st = 2;
          } else {
            exact_ac_step(s, T, row);
            st = z_block_done(s.z) ? 1 : 0;
          }
        }
      }
    }
    if (!__any_sync(0xffffffffu, st == 1)) break;
    {
      if (st == 1 && s.z > 64u) {  // what ended the block?
        if (z_no_code(s.z)) {
          exact_ac_undo_no_code(s);
          st = 2;
        } else if (z_overrun(s.z)) {
          err = HCJ_DEV_COEF_INDEX;
          *err_pos = s.br.pos;
          st = 3;
        }
      }
      const bool have = st == 1 && s.z != 0u;  // a finished block in the lane's row
      if (have && exact_share_may_be_wide(s) && exact_share(s, T, row) >= (uint32_t)HCJ_WIDE_SHARE) flag_wide_block(sc, s.blk);
      warp_store_full(__ballot_sync(0xffffffffu, have), s.blk, stage, lane, coefs);
      if (have) exact_next_block(s, T, bpm);
      if (st == 1) {
        if (s.blk + 1 >= in.nblocks_end || s.br.pos >= lim || (s.c == 0u && s.br.pos >= in.hi)) st = 2;
        else st = exact_dc_step(s, T, row) ? 0 : 2;
      }
    }
  }
  // the literal loop keeps the exact share of the block in progress
  if (entered && st == 2 && s.z != 0u) s.share = exact_share(s, T, row);
  if (entered) {
    exact_save_pred(s);
    in.p = s.br.pos;
    in.cz = (s.c << 8) | s.z;
    in.blk = s.blk;
    in.pred[0] = s.p0, in.pred[1] = s.p1, in.pred[2] = s.p2, in.pred[3] = s.p3;
    in.share = s.share;
    if (err) {  // the lane is done: leave its row clean for the next pass of this warp
      in.valid = false;
      uint4 *src = reinterpret_cast<uint4 *>(row);
#pragma unroll
      for (int j = 0; j < 8; j++) src[j] = make_uint4(0u, 0u, 0u, 0u);
    }
  }
  return err;
}

__device__ __forceinline__ int warp_exact_pass(const ScanCtx &sc, const SmemTables &st, const Local L, uint32_t *stage,
                                               int lane, const PassIn &in, int16_t *coefs, uint32_t *err_pos) {
  uint32_t *coefs32 = reinterpret_cast<uint32_t *>(coefs);
  const uint32_t bpm = sc.bpm;
  uint32_t c = in.cz >> 8, z = in.cz & 0xffu, share = in.share;
  int32_t blk = in.blk;
  bool active = in.valid;
  uint32_t comp = st.blk_comp[c];
  Tables t = sc.tab[comp];
  const uint32_t stage_sa = (uint32_t)__cvta_generic_to_shared(stage);
  const uint32_t mine_sa = stage_sa + (uint32_t)lane * HR_ROW_WORDS * 4u;
  const uint32_t quant_sa = (uint32_t)__cvta_generic_to_shared(st.quant);
  uint32_t q_sa = quant_sa + comp * 512u;
  int32_t p0 = in.pred[0], p1 = in.pred[1], p2 = in.pred[2], p3 = in.pred[3];
  int32_t pcur = comp == 0u ? p0 : comp == 1u ? p1 : comp == 2u ? p2 : p3;
  BitReader br;
  br.init(sc.words, in.p, active ? in.end_bits : 0u);
  int err = HCJ_DEV_OK;

  while (__any_sync(0xffffffffu, active)) {
    bool done_blk = false;
    if (active) {
      const bool isdc = z == 0u;
      if (isdc && ((c == 0u && br.pos >= in.hi && br.pos < in.end_bits) || blk + 1 >= in.nblocks_end)) {
        active = false;
      } else {
        const Symbol s = read_symbol(br, L, t, isdc);
        if (s.e == 0u) {
          err = isdc ? HCJ_DEV_NO_DC_CODE : HCJ_DEV_NO_AC_CODE;
          active = false;
        } else {
          br.skip(s.nbits);
          const bool eob = !isdc && (s.e & 0xffu) == 0u;
          const uint32_t zi = isdc ? 0u : z + s.run;
          if (zi >= 64u && !eob) {
            err = HCJ_DEV_COEF_INDEX;
            active = false;
          } else {
            pcur += isdc ? s.value : 0;
            const int32_t v = isdc ? pcur : s.value;
            blk += isdc ? 1 : 0;
            if (isdc && (pcur < -32768 || pcur > 32767)) {
              err = HCJ_DEV_DC_RANGE;
              active = false;
            }
            if (isdc || (s.size != 0u && !eob)) {
              asm volatile("st.shared.u16 [%0], %1;" ::"r"(mine_sa + zi * 2u), "h"((short)v) : "memory");
              int32_t qv;
              asm volatile("ld.shared.s32 %0, [%1];" : "=r"(qv) : "r"(q_sa + zi * 4u));
              share += (uint32_t)(v < 0 ? -v : v) * (uint32_t)qv;
            }
            z = eob ? 64u : zi + 1u;
            if (z >= 64u && active) {
              done_blk = true;
              if (share >= (uint32_t)HCJ_WIDE_SHARE) flag_wide_block(sc, blk);
              share = 0;
              z = 0;
              p0 = comp == 0u ? pcur : p0;
              p1 = comp == 1u ? pcur : p1;
              p2 = comp == 2u ? pcur : p2;
              p3 = comp == 3u ? pcur : p3;
              c = c + 1u == bpm ? 0u : c + 1u;
              comp = st.blk_comp[c];
              pcur = comp == 0u ? p0 : comp == 1u ? p1 : comp == 2u ? p2 : p3;
              t = sc.tab[comp];
              q_sa = quant_sa + comp * 512u;
            }
          }
        }
      }
    }
    // write out the blocks completed in this step: one 128-byte line per block, all lanes cooperating
    uint32_t mask = __ballot_sync(0xffffffffu, done_blk);
    while (mask) {
      const int l = __ffs((int)mask) - 1;
      mask &= mask - 1u;
      const int32_t bidx = __shfl_sync(0xffffffffu, blk, l);
      const uint32_t sa = stage_sa + ((uint32_t)l * HR_ROW_WORDS + (uint32_t)lane) * 4u;
      uint32_t w;
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(sa) : "memory");
      asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(0u) : "memory");
      coefs32[(size_t)bidx * 32 + lane] = w;
    }
  }
  // a lane stops in the middle of a block only when the model raises there: the block is not written (the image's
  // status says so); leave the stage clean for the next pass of this warp
  if (z != 0u && in.valid) {
    for (uint32_t w = 0; w < 32u; w++) asm volatile("st.shared.u32 [%0], %1;" ::"r"(mine_sa + w * 4u), "r"(0u) : "memory");
  }
  *err_pos = br.pos;
  return err;
}

constexpr int HR_THREADS = 512;

// The exact pass of one restart interval per lane (same symbol semantics as subseq_write), with the
// coefficient block of every lane staged in shared memory and written out by the whole warp as one
// 128-byte line when it completes: scattered 2-byte stores cost one L2 partial-sector transaction per
// symbol and were the bottleneck of this kernel.
__global__ void __launch_bounds__(HR_THREADS, 2) k_huff_restart(DecodeBatchDev b) {
  extern __shared__ uint4 s_dyn4[];
  SmemTables &st = *reinterpret_cast<SmemTables *>(s_dyn4);
  ScanCtx &sc = *reinterpret_cast<ScanCtx *>(reinterpret_cast<char *>(s_dyn4) + ((sizeof(SmemTables) + 15) & ~size_t(15)));
  uint32_t *s_stage = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(&sc) + ((sizeof(ScanCtx) + 15) & ~size_t(15)));

  const uint32_t img = b.list_restart[blockIdx.y + b.lr_lo];
  const HcjImageDesc &d = b.descs[img];
  const uint32_t seg = blockIdx.x * HR_THREADS + threadIdx.x;
  if (blockIdx.x * HR_THREADS >= d.nseg_expected) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t *stage = s_stage + warp * HR_STAGE_WORDS;
  for (int j = lane; j < HR_STAGE_WORDS; j += 32) stage[j] = 0u;
  const FastTables T = load_tables(st, s_stage + (HR_THREADS / 32) * HR_STAGE_WORDS, b, d);
  __syncthreads();
  fill_scan_ctx(sc, st, b, d, 0);
  __syncthreads();
  HcjImageState *state = b.states + img;
  const Local L{T, st.quant, st.blk_comp};
  const bool valid = seg < d.nseg_expected && state->status == 0;

  const uint32_t *segs = b.seg_offs + d.seg_off;
  const uint32_t seg_begin = valid ? segs[seg] : 0u, seg_end = valid ? segs[seg + 1] : 0u;
  const uint32_t seg_bits = (seg_end - seg_begin) * 8u;
  const uint32_t ri = d.ri ? d.ri : d.nmcu;
  const uint32_t mcu0 = min(seg * ri, d.nmcu), mcu1 = min(mcu0 + ri, d.nmcu);
  const uint32_t bpm = d.bpm;
  int16_t *coefs = b.coefs + d.coef_off * 64;

  if (valid && seg_bits <= 16u) {
    // Degenerate interval: the model's `show` bound (bitstream_reader.ml:32) is in play; decode it with
    // the literal per-block routine and direct stores.
    BitReader br;
    br.init(sc.words, seg_begin * 8u, seg_end * 8u);
    int32_t p0 = 0, p1 = 0, p2 = 0, p3 = 0;
    int64_t blk = (int64_t)mcu0 * bpm;
    for (uint32_t mcu = mcu0; mcu < mcu1; mcu++) {
      for (uint32_t k = 0; k < bpm; k++, blk++) {
        const uint32_t comp = st.blk_comp[k];
        int32_t pred = comp == 0 ? p0 : comp == 1 ? p1 : comp == 2 ? p2 : p3;
        int err = decode_block_exact(br, L, sc.tab[comp], seg_bits, pred, coefs + blk * 64);
        flag_wide_block(sc, blk);
        if (err) {
          raise_status(state, err, br.pos);
          mcu = mcu1;
          break;
        }
        if (comp == 0) p0 = pred;
        else if (comp == 1) p1 = pred;
        else if (comp == 2) p2 = pred;
        else p3 = pred;
      }
    }
  }

  // ---- warp-synchronous exact pass over the interval
  PassIn in;
  in.valid = valid && seg_bits > 16u && mcu1 > mcu0;
  in.p = seg_begin * 8u;
  in.cz = 0u;
  in.hi = 0xffffffffu;
  in.end_bits = seg_end * 8u;
  in.blk = (int32_t)(mcu0 * bpm) - 1;
  in.pred[0] = in.pred[1] = in.pred[2] = in.pred[3] = 0;
  in.nblocks_end = (int32_t)(mcu1 * bpm);
  in.share = 0;
  uint32_t err_pos = 0;
  int err = warp_exact_fast(sc, T, stage, lane, in, coefs, &err_pos);
  if (err) raise_status(state, err, err_pos);
  err = warp_exact_pass(sc, st, L, stage, lane, in, coefs, &err_pos);
  if (err) raise_status(state, err, err_pos);
}

void launch_huff_restart(const DecodeBatchDev &b, cudaStream_t s) {
  if (b.lr_hi <= b.lr_lo) return;
  const size_t smem = ((sizeof(SmemTables) + 15) & ~size_t(15)) + ((sizeof(ScanCtx) + 15) & ~size_t(15)) +
                      (HR_THREADS / 32) * HR_STAGE_WORDS * sizeof(uint32_t) + lut_smem_bytes(b);
  dim3 grid((b.max_segments + HR_THREADS - 1) / HR_THREADS, b.lr_hi - b.lr_lo);
  k_huff_restart<<<grid, HR_THREADS, smem, s>>>(b);
}

// ================================================================================================
// K3: self-synchronising speculative subsequence decode, for scans without restart markers (the reference encoder's
// own format) and for scans whose restart intervals are long (a camera's "one MCU row per interval", an interval that
// spans the image): north_star's "in parallel across restart intervals, and within an interval".
//
// The UNIT of the decoder is a run of entropy-coded bits that starts byte aligned with all DC predictors at zero and
// holds a known range of blocks: the whole scan, or one restart interval (bytes [segs[u], segs[u + 1]) of the image's
// destuffed data, MCUs [u * ri, (u + 1) * ri)).  A unit is decoded exactly as the model decodes a scan of its own: bits
// beyond its end read as zero, its blocks are decoded whatever the bits say (decoder.ml:118-165,347-397).  Every unit
// is cut into subsequences of sub_bits bits (chosen per image on the host); the subsequences of an image are numbered
// through all its units (k_spec_units: prefix sums of the units' subsequence counts), so that the grids below are
// full whatever the number of images and units.  A decoder state between symbols is (bit position, block-in-MCU,
// zig-zag index), 16 bits packed relative to the subsequence boundary.
//   k_spec_units   (only if the launch holds images with restart intervals) subsequence counts of the units
//   k_spec_sync    one thread per subsequence: decodes the guess_bits bits in front of it from a guessed state (block
//                  0 of an MCU, DC next) - a decoder started from a guess is in step with the real one after a couple
//                  of MCUs - and then the subsequence itself from the state that leaves it in, counting the blocks it
//                  begins and the DC differentials per component; AC symbols go several per look-up
//                  (multi_sync_entry).  The first subsequence of a unit starts from the exact state.
//   k_spec_fix     one CTA per image: fix-point rounds over the subsequences whose left neighbour's end state differs
//                  from the start state they used (a compacted list; almost always empty); the first subsequence
//                  of a unit is exact, so after k rounds the first k + 1 are and it terminates for any input.  Then
//                  segmented exclusive scans of (blocks begun, DC sums per component) give every subsequence its
//                  first block index and DC predictors, and the blocks shared by two threads are cleared;
//   k_spec_write   the exact pass: stores the coefficients (warp_exact_fast + warp_exact_pass).
// Undefined codes / overlong runs met while speculating are skipped deterministically (subseq_sync); only
// the exact pass reports them.  Units of <= 16 bits, where the model's `show` bound is observable, are
// decoded serially with the literal per-block routine (k_spec_fix).
// ================================================================================================
constexpr int SPEC_THREADS = 256;
constexpr int SPEC_WRITE_THREADS = 512;  // the exact pass: same shape as K2 (2 CTAs of 16 warps per SM at 64 registers)

__device__ __forceinline__ uint32_t spec_pack(uint32_t p, uint32_t base, uint32_t cz) {
  return ((p - base) << 10) | ((cz >> 8) << 6) | (cz & 63u);
}
__device__ __forceinline__ void spec_unpack(uint32_t s, uint32_t base, uint32_t &p, uint32_t &cz) {
  p = base + (s >> 10);
  cz = (((s >> 6) & 15u) << 8) | (s & 63u);
}

// The multi-symbol form of the image's AC tables (multi_sync_entry), behind the single-symbol tables in shared memory.
// Call between two barriers: reads what load_tables wrote.
__device__ __forceinline__ void build_multi_tables(FastTables &T, const DecodeBatchDev &b, const HcjImageDesc &d) {
  uint32_t *multi = const_cast<uint32_t *>(T.sub) + (size_t)b.max_pairs * 2 * LUT_SUB_ENTRIES;
  const uint32_t npairs = b.table_sets[d.table_set].npairs;
  for (uint32_t i = threadIdx.x; i < npairs * HCJ_LUT_SIZE; i += blockDim.x) {
    const uint32_t pr = i >> HCJ_LUT_BITS;
    multi[i] = multi_sync_entry(T.fast + (pr * 2 + 1) * HCJ_LUT_SIZE, i & (HCJ_LUT_SIZE - 1));
  }
  T.multi = multi;
}
static inline size_t multi_smem_bytes(const DecodeBatchDev &b) { return (size_t)b.max_pairs * HCJ_LUT_SIZE * sizeof(uint32_t); }

// Synchronisation decode of one subsequence per lane (the semantics of subseq_sync): the fast steps run
// warp-synchronously with the per-block work batched as in warp_exact_fast; the literal loop finishes
// what is left (the last 32 bits of the unit, undefined codes met while speculating).
template <bool MULTI = true>
__device__ __forceinline__ void warp_subseq_sync(const ScanCtx &sc, const Local L, bool valid, uint32_t p, uint32_t cz,
                                                 uint32_t hi, uint32_t end_bits, SubResult &r, int32_t *dpre) {
  const FastTables T = L.ft;
  const uint32_t bpm = sc.bpm;
  const uint32_t lim = min(hi, end_bits >= 32u ? end_bits - 32u : 0u);
  const uint32_t lim_m = min(lim, hi >= (uint32_t)HCJ_LUT_BITS ? hi - (uint32_t)(HCJ_LUT_BITS - 1) : 0u);
  SyncLane s;
  s.c = cz >> 8;
  s.z = cz & 0xffu;
  s.nstart = 0;
  s.d0 = s.d1 = s.d2 = s.d3 = 0;
  s.first_p = 0xffffffffu;
  s.nbefore = 0;
  const bool entered = valid && p < lim;
  s.br.init(sc.words, entered ? p : 0u);
  s.br.pos = p;
  sync_bind_block(s, T);
  int st = !entered ? 2 : s.z != 0u ? 0 : 1;  // 0 = mid-block, 1 = at a block boundary, 2 = left
  // Unlike the exact pass, the per-block code is light here (no write-out), and when decoding from a
  // guessed state the "blocks" of the lanes are of wildly different lengths: lanes at a block boundary are
  // served as soon as a quarter of the running lanes are waiting (measured against a half and an eighth).
#ifndef HCJ_SYNC_THR
#define HCJ_SYNC_THR 2
#endif
#ifndef HCJ_SYNC_UNROLL
#define HCJ_SYNC_UNROLL 2
#endif
  const int thr = HCJ_SYNC_THR;
  for (;;) {
#pragma unroll
    for (int u = 0; u < HCJ_SYNC_UNROLL; u++) {
      if (st == 0) {
        if (s.br.pos >= lim) {
          st = 2;
        } else {
          if (MULTI) sync_ac_step_multi(s, T, lim_m);
          else sync_ac_step_single(s, T);
          st = z_block_done(s.z) ? 1 : 0;
        }
      }
    }
    const uint32_t wmask = __ballot_sync(0xffffffffu, st == 1);
    const uint32_t smask = __ballot_sync(0xffffffffu, st == 0);
    if ((wmask | smask) == 0u) break;
    if (wmask != 0u && (smask == 0u || (__popc(wmask) << thr) >= __popc(wmask | smask))) {
      if (st == 1) {
        if (s.z != 0u) sync_next_block(s, T, bpm);
        if (s.br.pos >= lim) {
          st = 2;
        } else {
          sync_dc_step(s, T, dpre);
          st = s.z != 0u ? 0 : 1;  // (an undefined code: one bit was skipped, still at the boundary)
        }
      }
    }
  }
  r.p = s.br.pos;
  r.cz = (s.c << 8) | s.z;
  r.nstart = s.nstart;
  r.dcsum[0] = s.d0, r.dcsum[1] = s.d1, r.dcsum[2] = s.d2, r.dcsum[3] = s.d3;
  r.first_p = s.first_p, r.nbefore = s.nbefore;
  if (valid && s.br.pos < hi) {
    SubResult r2;
    int32_t dpre2[HCJ_MAX_COMP];
    subseq_sync(sc, L, s.br.pos, r.cz, hi, r2, end_bits, dpre2);
    r.p = r2.p;
    r.cz = r2.cz;
    if (r.first_p == 0xffffffffu && r2.first_p != 0xffffffffu) {
      r.first_p = r2.first_p, r.nbefore = r.nstart + r2.nbefore;
#pragma unroll
      for (int k = 0; k < HCJ_MAX_COMP; k++) dpre[k] = r.dcsum[k] + dpre2[k];
    }
    r.nstart += r2.nstart;
#pragma unroll
    for (int k = 0; k < HCJ_MAX_COMP; k++) r.dcsum[k] += r2.dcsum[k];
  }
}

// What every K3 kernel needs about its image.  Returns false if there is nothing to do for this CTA.
struct SpecImage {
  const HcjImageDesc *d;
  HcjImageState *state;
  uint32_t S, nunits, nsub;  // subsequence length; units; subsequences of all units
  const uint32_t *segs;      // unit u = bytes [segs[u], segs[u + 1]) of the image's entropy data
  const uint32_t *unit_sub;  // nunits > 1: index of every unit's first subsequence (nunits + 1 entries, k_spec_units)
  uint16_t *start, *end2;
  uint32_t *first;           // where the first MCU begun in the subsequence starts (spec_pack_first)
  int32_t *nstart, *blk;     // blocks begun in the subsequence; index of the first of them (k_spec_fix)
  int4 *dc, *dpre;           // DC sums per component of the subsequence / of its part in front of that first MCU
};
// position (relative to the subsequence's first bit: < 2^15) of the first MCU begun and the blocks begun before it (< 16);
// bit 31: none
__device__ __forceinline__ uint32_t spec_pack_first(const SubResult &r, uint32_t lo) {
  return r.first_p == 0xffffffffu ? 0x80000000u : (r.first_p - lo) | (r.nbefore << 16);
}
__device__ __forceinline__ uint32_t spec_unit_subs(uint32_t bits, uint32_t S) { return bits <= 16u ? 0u : (bits + S - 1u) / S; }
__device__ __forceinline__ bool spec_image(const DecodeBatchDev &b, uint32_t list_index, SpecImage &si) {
  const uint32_t img = b.list_spec[list_index + b.ls_lo];
  si.d = &b.descs[img];
  si.state = b.states + img;
  if (si.state->status != 0) return false;
  si.S = si.d->sub_bits;
  si.nunits = si.d->nseg_expected;
  si.segs = b.seg_offs + si.d->seg_off;
  si.unit_sub = b.seg_sub + si.d->seg_off;
  si.nsub = si.nunits > 1u ? si.unit_sub[si.nunits] : spec_unit_subs(si.state->ent_len * 8u, si.S);
  si.start = b.sub_start + si.d->sub_off;
  si.end2 = b.sub_end2 + si.d->sub_off;
  si.first = b.sub_first + si.d->sub_off;
  si.nstart = b.sub_nstart + si.d->sub_off;
  si.blk = b.sub_blk + si.d->sub_off;
  si.dc = b.sub_dc + si.d->sub_off;
  si.dpre = b.sub_dpre + si.d->sub_off;
  return true;
}

// Subsequence j of the image: its unit, its place in it and the unit's block range.
struct SpecSub {
  uint32_t jl;             // index within the unit
  uint32_t lo, hi;         // bits [lo, hi) of the image's entropy data
  uint32_t ulo, uend;      // the unit's bits
  bool last;               // last subsequence of the unit
  int32_t blk0, blk_end;   // the unit's blocks
};
__device__ __forceinline__ SpecSub spec_sub(const SpecImage &si, uint32_t j) {
  SpecSub q;
  uint32_t u = 0, first = 0, count = si.nsub;
  if (si.nunits > 1u) {
    uint32_t lo = 0, hi = si.nunits;  // largest u with unit_sub[u] <= j (units without subsequences share their successor's entry)
    while (hi - lo > 1u) {
      const uint32_t mid = (lo + hi) >> 1;
      if (__ldg(si.unit_sub + mid) <= j) lo = mid;
      else hi = mid;
    }
    u = lo;
    first = __ldg(si.unit_sub + u);
    count = __ldg(si.unit_sub + u + 1) - first;
  }
  const HcjImageDesc &d = *si.d;
  q.jl = j - first;
  q.ulo = (si.nunits > 1u ? __ldg(si.segs + u) : 0u) * 8u;
  q.uend = (si.nunits > 1u ? __ldg(si.segs + u + 1) : si.state->ent_len) * 8u;
  q.lo = q.ulo + q.jl * si.S;
  q.hi = min(q.lo + si.S, q.uend);
  q.last = q.jl + 1u == count;
  const uint32_t ri = d.ri ? d.ri : d.nmcu;
  const uint32_t mcu0 = min(u * ri, d.nmcu), mcu1 = min(mcu0 + ri, d.nmcu);
  q.blk0 = (int32_t)(mcu0 * (uint32_t)d.bpm);
  q.blk_end = (int32_t)(mcu1 * (uint32_t)d.bpm);
  return q;
}

// grid: images of the launch's list_spec.  Exclusive prefix sums of the units' subsequence counts.
__global__ void __launch_bounds__(SPEC_THREADS) k_spec_units(DecodeBatchDev b) {
  __shared__ uint32_t s_warp[SPEC_THREADS / 32];
  const uint32_t img = b.list_spec[blockIdx.x + b.ls_lo];
  const HcjImageDesc &d = b.descs[img];
  if (d.nseg_expected <= 1u || b.states[img].status != 0) return;
  const uint32_t *segs = b.seg_offs + d.seg_off;
  uint32_t *unit_sub = b.seg_sub + d.seg_off;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  uint32_t carry = 0;
  for (uint32_t u0 = 0; u0 < d.nseg_expected; u0 += SPEC_THREADS) {
    const uint32_t u = u0 + t;
    const uint32_t v = u < d.nseg_expected ? spec_unit_subs((segs[u + 1] - segs[u]) * 8u, d.sub_bits) : 0u;
    const uint32_t incl = warp_incl_scan(v, lane);
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t base = 0, total = 0;
#pragma unroll
    for (int k = 0; k < SPEC_THREADS / 32; k++) {
      const uint32_t x = s_warp[k];
      if (k < warp) base += x;
      total += x;
    }
    if (u < d.nseg_expected) unit_sub[u] = carry + base + incl - v;
    carry += total;
  }
  if (t == 0) unit_sub[d.nseg_expected] = carry;
}

// One value of the segmented scans of k_spec_fix: blocks begun and DC sums per component of a subsequence; `flag` =
// it is the first one of its unit (the sums start again from the unit's first block and predictors 0).
struct SegVal {
  int32_t v[5];
  uint32_t flag;
};
__device__ __forceinline__ void seg_combine(SegVal &right, const SegVal &left) {  // right = left (+) right
  if (!right.flag) {
#pragma unroll
    for (int k = 0; k < 5; k++) right.v[k] += left.v[k];
  }
  right.flag |= left.flag;
}

// The image-wide step between the synchronisation decode and the exact pass: one small CTA per image.  The step is
// bound by the latency of a handful of lanes decoding a subsequence each (a round takes as long as one subsequence
// takes one lane), so what matters is how many images are in flight per SM: 128 threads and no more shared memory
// than the single-symbol tables (8 CTAs per SM).  (Run as the tail of the image's last k_spec_sync CTA instead - tables already loaded, no launch -
// it took the same time in total: 2.64 ms against 1.95 + 0.65 ms; the CTA slots are the bottleneck, not the issue
// slots.)
constexpr int SPEC_FIX_THREADS = 128;
__global__ void __launch_bounds__(SPEC_FIX_THREADS, 8) k_spec_fix(DecodeBatchDev b) {
  extern __shared__ uint4 s_dyn4[];
  SmemTables &st = *reinterpret_cast<SmemTables *>(s_dyn4);
  ScanCtx &sc = *reinterpret_cast<ScanCtx *>(reinterpret_cast<char *>(s_dyn4) + ((sizeof(SmemTables) + 15) & ~size_t(15)));
  void *lut_smem = reinterpret_cast<char *>(&sc) + ((sizeof(ScanCtx) + 15) & ~size_t(15));
  __shared__ SegVal s_seg[SPEC_FIX_THREADS / 32];
  __shared__ uint32_t s_count;
  SpecImage si;
  if (!spec_image(b, blockIdx.x, si)) return;
  const HcjImageDesc &d = *si.d;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  int16_t *coefs = b.coefs + d.coef_off * 64;
  const int n = (int)si.nsub;
  uint32_t *list = b.sub_list + d.sub_off;

  // ---- which subsequences were decoded from a state that is not their left neighbour's end state?
  auto collect = [&]() {
    if (t == 0) s_count = 0;
    __syncthreads();
    for (int j0 = 0; j0 < n; j0 += SPEC_FIX_THREADS) {
      const int j = j0 + t;
      // (the first subsequence of a unit has the packed start state 0 and no left neighbour: its `start` entry is
      // compared with the end of the previous unit's last subsequence only if jl > 0)
      bool need = false;
      if (j >= 1 && j < n && __ldcg(si.end2 + j - 1) != __ldcg(si.start + j)) need = si.nunits <= 1u || spec_sub(si, (uint32_t)j).jl > 0u;
      const uint32_t mask = __ballot_sync(0xffffffffu, need);
      if (mask) {
        uint32_t at = 0;
        if (lane == 0) at = atomicAdd(&s_count, (uint32_t)__popc(mask));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (need) list[at + __popc(mask & ((1u << lane) - 1u))] = (uint32_t)j;
      }
    }
    __syncthreads();
    return (int)s_count;
  };
  int nredo = collect();
  uint32_t rounds = 0, redone = 0;  // diagnostics (HcjImageState::pad_, printed under HCJ_SPEC_STATS)
  // units of <= 16 bits (the model's `show` bound, bitstream_reader.ml:32, is in play): decoded serially below
  bool tiny = false;
  for (uint32_t u = t; u < si.nunits; u += SPEC_FIX_THREADS) tiny = tiny || (si.segs[u + 1] - si.segs[u]) * 8u <= 16u;
  if (si.nunits == 1u) tiny = si.state->ent_len * 8u <= 16u;
  const bool any_tiny = __syncthreads_or(tiny);

  if (nredo || any_tiny) {  // CTA-uniform; the tables are only loaded now
    const FastTables T = load_tables(st, lut_smem, b, d);
    __syncthreads();
    fill_scan_ctx(sc, st, b, d, si.state->ent_len * 8u);
    __syncthreads();
    const Local LT{T, st.quant, st.blk_comp};
    if (any_tiny) {
      const uint32_t ri = d.ri ? d.ri : d.nmcu;
      for (uint32_t u = t; u < si.nunits; u += SPEC_FIX_THREADS) {
        const uint32_t b0 = si.nunits > 1u ? si.segs[u] : 0u, b1 = si.nunits > 1u ? si.segs[u + 1] : si.state->ent_len;
        const uint32_t bits = (b1 - b0) * 8u;
        if (bits > 16u) continue;
        BitReader br;
        br.init(sc.words, b0 * 8u, b1 * 8u);
        int32_t pred[HCJ_MAX_COMP] = {0, 0, 0, 0};
        const uint32_t mcu0 = min(u * ri, d.nmcu), mcu1 = min(mcu0 + ri, d.nmcu);
        for (int64_t blk = (int64_t)mcu0 * d.bpm; blk < (int64_t)mcu1 * d.bpm; blk++) {
          const uint32_t comp = st.blk_comp[blk % d.bpm];
          const int err = decode_block_exact(br, LT, sc.tab[comp], bits, pred[comp], coefs + blk * 64);
          flag_wide_block(sc, blk);
          if (err) {
            raise_status(si.state, err, br.pos);
            break;
          }
        }
      }
    }
    // ---- fix-point rounds over the compacted list
    while (nredo) {
      rounds++;
      redone += (uint32_t)nredo;
      for (int k0 = 0; k0 < nredo; k0 += SPEC_FIX_THREADS) {
        const int k = k0 + t;
        const bool valid = k < nredo;
        const uint32_t j = valid ? __ldcg(list + k) : 1u;
        const uint32_t ns = __ldcg(si.end2 + j - 1);  // reads within a round are unsynchronised (chaotic relaxation): the fix-point is unique
        const SpecSub q = spec_sub(si, min(j, (uint32_t)n - 1u));
        uint32_t p, cz;
        spec_unpack(ns, q.lo, p, cz);
        SubResult r;
        warp_subseq_sync<false>(sc, LT, valid, p, cz, q.hi, q.uend, r, reinterpret_cast<int32_t *>(si.dpre + j));
        if (valid) {
          si.start[j] = (uint16_t)ns;
          si.end2[j] = (uint16_t)spec_pack(r.p, q.hi, r.cz);
          si.first[j] = spec_pack_first(r, q.lo);
          si.nstart[j] = (int32_t)r.nstart;
          si.dc[j] = make_int4(r.dcsum[0], r.dcsum[1], r.dcsum[2], r.dcsum[3]);
        }
      }
      __syncthreads();
      nredo = collect();
    }
  }

  if (t == 0) si.state->pad_ = min(rounds, 255u) | (redone << 8);
  // ---- segmented exclusive scans over the image's subsequences, in place: index of the first block begun in every
  // subsequence (a unit's count starts at its first block) and the DC predictors there.
  SegVal carry;
#pragma unroll
  for (int k = 0; k < 5; k++) carry.v[k] = 0;
  carry.flag = 0;
  for (int j0 = 0; j0 < n; j0 += SPEC_FIX_THREADS) {
    const int j = j0 + t;
    SegVal own, x;
#pragma unroll
    for (int k = 0; k < 5; k++) own.v[k] = 0;
    own.flag = 0;
    if (j < n) {
      const int4 dc = __ldcg(si.dc + j);
      own.v[0] = __ldcg(si.nstart + j), own.v[1] = dc.x, own.v[2] = dc.y, own.v[3] = dc.z, own.v[4] = dc.w;
      if (si.nunits > 1u) {
        const SpecSub q = spec_sub(si, (uint32_t)j);
        own.flag = q.jl == 0u;
        x = own;
        if (own.flag) x.v[0] += q.blk0;
      } else {
        own.flag = j == 0;
        x = own;
      }
    } else {
      x = own;
    }
    // inclusive segmented scan of x inside the warp
#pragma unroll
    for (int dlt = 1; dlt < 32; dlt <<= 1) {
      SegVal o;
#pragma unroll
      for (int k = 0; k < 5; k++) o.v[k] = __shfl_up_sync(0xffffffffu, x.v[k], dlt);
      o.flag = __shfl_up_sync(0xffffffffu, x.flag, dlt);
      if (lane >= dlt) seg_combine(x, o);
    }
    __syncthreads();  // s_seg may still be read from the previous chunk
    if (lane == 31) s_seg[warp] = x;
    __syncthreads();
    SegVal before = carry, total = carry;  // everything before this warp / the whole chunk, carried from chunk to chunk
    for (int k = 0; k < SPEC_FIX_THREADS / 32; k++) {
      SegVal w = s_seg[k];
      seg_combine(w, total);
      total = w;
      if (k + 1 == warp) before = w;
    }
    seg_combine(x, before);
    carry = total;
    carry.flag = 0;
    if (j < n) {
      si.blk[j] = x.v[0] - own.v[0];  // exclusive (si.nstart keeps the counts: k_spec_write sorts by them)
      si.dc[j] = make_int4(x.v[1] - own.v[1], x.v[2] - own.v[2], x.v[3] - own.v[3], x.v[4] - own.v[4]);
    }
  }
}

// Shared memory of k_spec_sync: [SmemTables][ScanCtx][tables][multi-symbol tables]
#ifndef HCJ_SPEC_SYNC_CTAS
#define HCJ_SPEC_SYNC_CTAS 4
#endif
__global__ void __launch_bounds__(SPEC_THREADS, HCJ_SPEC_SYNC_CTAS) k_spec_sync(DecodeBatchDev b) {
  extern __shared__ uint4 s_dyn4[];
  SmemTables &st = *reinterpret_cast<SmemTables *>(s_dyn4);
  ScanCtx &sc = *reinterpret_cast<ScanCtx *>(reinterpret_cast<char *>(s_dyn4) + ((sizeof(SmemTables) + 15) & ~size_t(15)));
  void *lut_smem = reinterpret_cast<char *>(&sc) + ((sizeof(ScanCtx) + 15) & ~size_t(15));
  SpecImage si;
  if (!spec_image(b, blockIdx.y, si)) return;
  if (blockIdx.x * SPEC_THREADS >= si.nsub) return;
  FastTables T = load_tables(st, lut_smem, b, *si.d);
  __syncthreads();
  build_multi_tables(T, b, *si.d);
  fill_scan_ctx(sc, st, b, *si.d, si.state->ent_len * 8u);
  __syncthreads();
  const Local LT{T, st.quant, st.blk_comp};

  const uint32_t j = blockIdx.x * SPEC_THREADS + threadIdx.x;
  const bool valid = j < si.nsub;
  const SpecSub q = spec_sub(si, valid ? j : 0u);
  // The state at the start of the subsequence: exact for the first one of a unit; for the others what a decoder
  // started guess_bits earlier from a guessed state is in when it gets here.  Where the guess had not yet fallen into
  // step, the left neighbour's end state will differ and k_spec_fix decodes the subsequence again.
  uint32_t p = q.lo, cz = 0;
  SubResult r;
  {
    const bool warm = valid && q.jl > 0u;
    const uint32_t p0 = q.lo - q.ulo > b.spec_guess_bits ? q.lo - b.spec_guess_bits : q.ulo;
    // (dpre: the DC sums in front of the first MCU start go straight to their place; the warm-up's are overwritten)
    int32_t *dpre = reinterpret_cast<int32_t *>(si.dpre + (valid ? j : 0u));
    warp_subseq_sync(sc, LT, warm, p0, 0u, q.lo, q.uend, r, dpre);
    if (warm) p = r.p, cz = r.cz;
    warp_subseq_sync(sc, LT, valid, p, cz, q.hi, q.uend, r, dpre);
  }
  if (valid) {
    si.start[j] = (uint16_t)spec_pack(p, q.lo, cz);
    si.end2[j] = (uint16_t)spec_pack(r.p, q.hi, r.cz);
    si.first[j] = spec_pack_first(r, q.lo);
    si.nstart[j] = (int32_t)r.nstart;
    si.dc[j] = make_int4(r.dcsum[0], r.dcsum[1], r.dcsum[2], r.dcsum[3]);
  }
}

// The exact pass: one thread per subsequence decodes the blocks that begin in it.
// (Sorting a CTA's subsequences by the number of blocks they begin, so that the lanes of a warp - which run in lock
// step block by block - get equal counts, and handing them to the warps in bundles from a shared counter was measured:
// 2.99 ms against 2.82 ms for this form on 1024 x 1080p; the same for K2's intervals sorted by length, 2.46 against
// 2.22 ms.  The lock step is lost inside the blocks, not at the end of the lanes' runs.)
// Shared memory: [SmemTables][ScanCtx][stage rows][tables]
__global__ void __launch_bounds__(SPEC_WRITE_THREADS, 2) k_spec_write(DecodeBatchDev b) {
  extern __shared__ uint4 s_dyn4[];
  SmemTables &st = *reinterpret_cast<SmemTables *>(s_dyn4);
  ScanCtx &sc = *reinterpret_cast<ScanCtx *>(reinterpret_cast<char *>(s_dyn4) + ((sizeof(SmemTables) + 15) & ~size_t(15)));
  uint32_t *s_stage = reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(&sc) + ((sizeof(ScanCtx) + 15) & ~size_t(15)));
  SpecImage si;
  if (!spec_image(b, blockIdx.y, si)) return;
  if (blockIdx.x * SPEC_WRITE_THREADS >= si.nsub) return;
  const HcjImageDesc &d = *si.d;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t *stage = s_stage + warp * HR_STAGE_WORDS;
  for (int k = lane; k < HR_STAGE_WORDS; k += 32) stage[k] = 0u;
  const FastTables T = load_tables(st, s_stage + (SPEC_WRITE_THREADS / 32) * HR_STAGE_WORDS, b, d);
  __syncthreads();
  fill_scan_ctx(sc, st, b, d, si.state->ent_len * 8u);
  __syncthreads();
  const Local LT{T, st.quant, st.blk_comp};
  int16_t *coefs = b.coefs + d.coef_off * 64;

  const uint32_t j = blockIdx.x * SPEC_WRITE_THREADS + threadIdx.x;
  PassIn in;
  in.valid = j < si.nsub;
  const uint32_t jj = in.valid ? j : 0u;
  const SpecSub q = spec_sub(si, jj);
  // the thread decodes the MCUs that begin in its subsequence (and finishes the last of them beyond its end)
  const uint32_t first = si.first[jj];
  in.valid = in.valid && (first >> 31) == 0u;
  in.p = q.lo + (first & 0xffffu);
  in.cz = 0u;
  const int4 dc = si.dc[jj], dpre = si.dpre[jj];
  in.pred[0] = dc.x + dpre.x, in.pred[1] = dc.y + dpre.y, in.pred[2] = dc.z + dpre.z, in.pred[3] = dc.w + dpre.w;
  in.blk = si.blk[jj] + (int32_t)((first >> 16) & 15u) - 1;
  in.hi = q.hi;  // (blocks that begin at or beyond the unit's end are decoded by the thread that gets there)
  in.end_bits = q.uend;
  in.nblocks_end = q.blk_end;
  in.share = 0;
  uint32_t err_pos = 0;
  int err = warp_exact_fast(sc, T, stage, lane, in, coefs, &err_pos);
  if (err) raise_status(si.state, err, err_pos);
  err = warp_exact_pass(sc, st, LT, stage, lane, in, coefs, &err_pos);
  if (err) raise_status(si.state, err, err_pos);
}

static inline size_t spec_base_smem(const DecodeBatchDev &b) {
  return ((sizeof(SmemTables) + 15) & ~size_t(15)) + ((sizeof(ScanCtx) + 15) & ~size_t(15)) + lut_smem_bytes(b);
}
void launch_huff_spec(const DecodeBatchDev &b, cudaStream_t s) {
  if (b.ls_hi <= b.ls_lo || b.max_sub_chunks == 0) return;
  const size_t base = spec_base_smem(b);
  const size_t smem_sync = base + multi_smem_bytes(b);
  const size_t smem_write = base + (SPEC_WRITE_THREADS / 32) * HR_STAGE_WORDS * sizeof(uint32_t);
  const dim3 grid(b.max_sub_chunks, b.ls_hi - b.ls_lo);
  if (b.spec_has_units) k_spec_units<<<b.ls_hi - b.ls_lo, SPEC_THREADS, 0, s>>>(b);
  k_spec_sync<<<grid, SPEC_THREADS, smem_sync, s>>>(b);
  k_spec_fix<<<b.ls_hi - b.ls_lo, SPEC_FIX_THREADS, base, s>>>(b);
  const dim3 grid_w((b.max_sub_chunks * SPEC_THREADS + SPEC_WRITE_THREADS - 1) / SPEC_WRITE_THREADS, b.ls_hi - b.ls_lo);
  k_spec_write<<<grid_w, SPEC_WRITE_THREADS, smem_write, s>>>(b);
}
int huff_spec_kernel_count(const DecodeBatchDev &b) { return 3 + (b.spec_has_units ? 1 : 0); }

// ================================================================================================
// K5: fused dequantise + inverse zig-zag + Chen IDCT + clip/level shift + store (+ crop).
//
// A CTA owns up to `tile_mcus` consecutive MCUs of one MCU row.  Their coefficient blocks are one
// contiguous run in HBM (block order = decode_seq order) and are staged into shared memory by ONE TMA tensor
// copy per tile (cp.async.bulk.tensor.2d, 128-byte swizzle: the per-thread 16-byte reads of a quarter-warp are
// bank-conflict free in a dense tile).  One thread reconstructs one 8x8 block entirely in registers; threads are ordered
// (component, block row, MCU, block column) so that a warp stores 32 horizontally adjacent blocks:
// every store instruction writes 256 contiguous bytes of one image row.
// ================================================================================================
constexpr int IDCT_MAX_THREADS = HCJ_IDCT_THREADS;

__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
  uint32_t sa = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

__device__ __forceinline__ void store_block_rows(const uint32_t pix[16], uint8_t *dst, int stride, int x, int y,
                                                 int w_limit, int h_limit) {
  // dst: plane base; (x, y): top-left sample of the block; samples outside w_limit x h_limit are cropped.
  uint8_t *row = dst + (size_t)y * stride + x;
  const bool fast = (x + 8 <= w_limit) && (((uintptr_t)row & 7u) == 0) && ((stride & 7) == 0);
  if (fast) {
#pragma unroll
    for (int r = 0; r < 8; r++)
      if (y + r < h_limit) *reinterpret_cast<uint2 *>(row + (size_t)r * stride) = make_uint2(pix[2 * r], pix[2 * r + 1]);
  } else {
#pragma unroll
    for (int r = 0; r < 8; r++) {
      if (y + r >= h_limit) break;
#pragma unroll
      for (int i = 0; i < 8; i++)
        if (x + i < w_limit) row[(size_t)r * stride + i] = (uint8_t)(pix[2 * r + (i >> 2)] >> (8 * (i & 3)));
    }
  }
}

// Rare path kept out of line so that its 64-bit temporaries do not cost the fast path registers.
__device__ __noinline__ void wide_block_store(const uint32_t *cw, const int32_t *q, uint8_t *dst, int stride, int x, int y,
                                              int w_limit, int h_limit) {
  uint32_t pix[16];
  reconstruct_wide(cw, q, pix);
  store_block_rows(pix, dst, stride, x, y, w_limit, h_limit);
}

// The same for a block of the staged (swizzled) tile: the coefficients are read again from shared memory, so that the
// fast path never has to keep its register copy addressable (a pointer to it would put all 32 words in local memory).
__device__ __noinline__ void wide_block_store_staged(const uint4 *tile, int slot, const int32_t *q, uint8_t *dst, int stride, int x,
                                                     int y, int w_limit, int h_limit) {
  uint32_t cw[32], pix[16];
  for (int j = 0; j < 8; j++) {
    const uint4 u = tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  reconstruct_wide(cw, q, pix);
  store_block_rows(pix, dst, stride, x, y, w_limit, h_limit);
}

// Scaled decode (HCJ_FLAG_SCALE_*): k x k samples (k = 4, 2, 1) of a block at (x, y) of its scaled plane, cropped like
// store_block_rows.  pix[r]: row r, packed.  With k = 4 a warp's 32 horizontally adjacent blocks write 128 contiguous bytes.
template <int K>
__device__ __forceinline__ void store_block_rows_k(const uint32_t *pix, uint8_t *dst, int stride, int x, int y, int w_limit,
                                                   int h_limit) {
  uint8_t *row = dst + (size_t)y * stride + x;
  const bool fast = (x + K <= w_limit) && (((uintptr_t)row & (K - 1)) == 0) && ((stride & (K - 1)) == 0);
#pragma unroll
  for (int r = 0; r < K; r++) {
    if (y + r >= h_limit) break;
    uint8_t *p = row + (size_t)r * stride;
    if (fast) {
      if (K == 4) *reinterpret_cast<uint32_t *>(p) = pix[r];
      else if (K == 2) *reinterpret_cast<uint16_t *>(p) = (uint16_t)pix[r];
      else *p = (uint8_t)pix[r];
    } else {
#pragma unroll
      for (int i = 0; i < K; i++)
        if (x + i < w_limit) p[i] = (uint8_t)(pix[r] >> (8 * i));
    }
  }
}

// Flagged blocks and 16-bit tables: the 64-bit column pass, out of line like wide_block_store_staged.
template <int K>
__device__ __noinline__ void scaled_block_store_wide(const uint4 *tile, int slot, const int32_t *q, uint8_t *dst, int stride, int x,
                                                     int y, int h_limit) {
  uint32_t cw[32], pix[K];
  for (int j = 0; j < 8; j++) {
    const uint4 u = tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  reconstruct_scaled(cw, q, K, true, pix);
  store_block_rows_k<K>(pix, dst, stride, x, y, stride, h_limit);
}

// One block of the staged tile reconstructed at 1/s (K = 8 / s) and stored.  K = 1 reads only the DC word.
template <int K>
__device__ __forceinline__ void scaled_block_store(const uint4 *tile, int slot, const int32_t *q, bool wide, uint8_t *dst, int stride,
                                                   int x, int y, int h_limit) {
  uint32_t pix[K];
  if (K == 1) {
    pix[0] = reconstruct_1x1(tile[slot * 8 + (slot & 7)].x, q[0]);  // chunk 0 of the block sits at chunk slot & 7 of its row
  } else if (wide) {
    scaled_block_store_wide<K>(tile, slot, q, dst, stride, x, y, h_limit);
    return;
  } else {
    uint32_t cw[32];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const uint4 u = tile[slot * 8 + (j ^ (slot & 7))];
      cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
    }
    reconstruct_scaled(cw, q, K, false, pix);
  }
  store_block_rows_k<K>(pix, dst, stride, x, y, stride, h_limit);
}

// HCJ_FLAG_LIBJPEG: one block of the staged tile reconstructed with libjpeg's islow IDCT and stored.  Flagged blocks and
// 16-bit tables take the 64-bit column pass out of line (islow_wide).
__device__ __noinline__ void islow_block_store_wide(const uint4 *tile, int slot, const int32_t *q, uint8_t *dst, int stride, int x,
                                                    int y, int h_limit) {
  uint32_t cw[32], pix[16];
  for (int j = 0; j < 8; j++) {
    const uint4 u = tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  islow_wide(cw, q, pix);
  store_block_rows(pix, dst, stride, x, y, stride, h_limit);
}

__device__ __forceinline__ void islow_block_store(const uint4 *tile, int slot, const int32_t *q, bool wide, uint8_t *dst, int stride,
                                                  int x, int y, int h_limit) {
  if (wide) {
    islow_block_store_wide(tile, slot, q, dst, stride, x, y, h_limit);
    return;
  }
  uint32_t cw[32], pix[16];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const uint4 u = tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  islow_fast(cw, q + 64, pix);
  store_block_rows(pix, dst, stride, x, y, stride, h_limit);
}

// Persistent CTAs (HCJ_IDCT_CTAS_PER_SM per SM): each owns a contiguous range of the batch's tiles and keeps the coefficient
// tile, the quant tables and the wide-block flags of tile i+1 in flight (cp.async) while tile i is being
// transformed.  The thread -> block mapping depends only on (image geometry, tile width): it is computed
// when either changes and kept in registers, so the per-tile overhead is a handful of instructions.
// mode: 0 = HCJ_OUT_YUV (cropped planes, packed), 1 = padded planes into b.out, 2 = padded planes into b.planes
constexpr int IDCT_Q_I32 = HCJ_MAX_COMP * 128;
constexpr int IDCT_FLAG_U4 = 3;  // 256 blocks = 8 flag words, at any alignment inside 3 x 16 bytes

// One pipeline stage in shared memory.  The tile is dense (128 bytes per block, no padding) and laid out by the
// TMA unit with its 128-byte swizzle: 16-byte chunk j of block r sits at chunk j ^ (r & 7) of row r, so the eight
// lanes of a quarter-warp, which read the same chunk of eight consecutive blocks, hit eight different bank groups.
struct alignas(1024) IdctStage {
  uint4 tile[IDCT_MAX_THREADS * 8];
  int32_t q[IDCT_Q_I32];
  uint4 flags[IDCT_FLAG_U4 + 1];
  uint64_t full;  // mbarrier: the TMA copies of the stage complete their bytes on it
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LAB_DONE;\n\t"
      "bra LAB_WAIT;\n"
      "LAB_DONE:\n\t}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk copy global -> shared (quant tables, flags)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 2-D tensor tile copy: the box of `map` whose first row is `row`
__device__ __forceinline__ void tma_tile_g2s(void *dst, const void *map, int32_t row, uint64_t *bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(0), "r"(row), "r"(smem_u32(bar))
      : "memory");
}

// The batch's tile plan: one 32-byte record per IDCT tile, image after image (HcjImageDesc::idct_tile_off), written
// by k_idct_plan before the transform.  With the plan in HBM the persistent CTAs do no per-tile geometry at all:
// thread 0 pulls the records two tiles ahead into shared memory (cp.async) and issues the loads from them.  (Walking
// the tiles with a cursor in thread 0 cost its warp ~130 instructions per tile on top of the ~1030 of the transform,
// and the other three warps waited for it at the tile barrier: profiles/r01s3_ncu_full_restart8_b296.csv.)
struct alignas(16) IdctTile {
  uint64_t blk0;     // first block of the tile in the batch coefficient buffer
  uint32_t img;      // image index
  uint32_t qt_off;   // the image's quant tables in the pool
  uint16_t my, m0;   // MCU row, first MCU
  uint16_t tm, nblk; // MCUs and blocks in the tile
  uint16_t qbytes;   // bytes of quant tables (512 per component)
  uint16_t remap;    // the thread -> block mapping differs from the previous tile's (first tile of an image, other width)
  uint32_t fused;    // RGB24 output: colour conversion inside the tile (HcjImageDesc::fused_rgb: 1 = 4:4:4, 2 = sub-sampled)
};
static_assert(sizeof(IdctTile) == 32, "two 16-byte cp.async per record");

size_t idct_plan_bytes(uint32_t tiles) { return ((size_t)tiles + 4) * sizeof(IdctTile); }
int idct_kernel_count() { return 2; }

__device__ __forceinline__ int idct_tile_width(const DecodeBatchDev &b, const HcjImageDesc &d, int &tiles_per_row) {
  const int tm_max = max(1, min(b.tile_mcus, IDCT_MAX_THREADS / d.bpm));
  tiles_per_row = (d.mcus_wide + tm_max - 1) / tm_max;
  return (d.mcus_wide + tiles_per_row - 1) / tiles_per_row;  // balanced tile width
}

// grid (ceil(max tiles of an image / 128), images of the launch)
__global__ void __launch_bounds__(128) k_idct_plan(DecodeBatchDev b) {
  const uint32_t img = b.img_lo + blockIdx.y;
  const HcjImageDesc &d = b.descs[img];
  const uint32_t tile = blockIdx.x * blockDim.x + threadIdx.x;
  if (!d.valid || tile >= d.idct_tiles) return;
  int tpr;
  const int tm_bal = idct_tile_width(b, d, tpr);
  const int my = (int)tile / tpr, tx = (int)tile - my * tpr;
  const int m0 = tx * tm_bal;
  const int tm = min(tm_bal, d.mcus_wide - m0);
  const int ptx = tx ? tx - 1 : tpr - 1;  // the tile before this one in the image
  const int ptm = min(tm_bal, d.mcus_wide - ptx * tm_bal);
  IdctTile t;
  t.blk0 = d.coef_off + ((uint64_t)my * d.mcus_wide + (uint64_t)m0) * d.bpm;
  t.img = img;
  t.qt_off = d.qt_off;
  t.my = (uint16_t)my;
  t.m0 = (uint16_t)m0;
  t.tm = (uint16_t)tm;
  t.nblk = (uint16_t)(tm * d.bpm);
  t.qbytes = (uint16_t)(d.ncomp * 512);
  t.remap = (uint16_t)(tile == 0 || tm != ptm);
  t.fused = d.fused_rgb;
  b.idct_plan[d.idct_tile_off + tile] = t;
}

// A thread's block inside the tile, valid for one (image geometry, tile width); kept in shared memory: the 64 values
// of a block need the registers, and what the compiler spills instead goes to local memory, which at 5 CTAs per SM
// does not fit the L1 that the tile stages leave (measured: 18 % of the kernel's stall samples were those reloads).
struct IdctMap {
  uint8_t *plane;      // the component's plane in the image's output / plane buffer
  int32_t stride;      // = crop width
  int32_t h_limit;
  uint32_t xy;         // sample offset of the block inside the tile's MCU row: x | y << 16
  uint32_t misc;       // staged block index | quant table << 8 | mine << 10 | wide << 11 | hs8 << 12 | vs8 << 18
};
// stored as two arrays (16 + 8 bytes per thread) so that a warp's reads are conflict free
struct IdctMapSmem {
  uint4 a[IDCT_MAX_THREADS];
  uint2 b[IDCT_MAX_THREADS];
  __device__ __forceinline__ void put(int t, const IdctMap &m) {
    const uint64_t p = reinterpret_cast<uint64_t>(m.plane);
    a[t] = make_uint4((uint32_t)p, (uint32_t)(p >> 32), (uint32_t)m.stride, (uint32_t)m.h_limit);
    b[t] = make_uint2(m.xy, m.misc);
  }
  __device__ __forceinline__ IdctMap get(int t) const {
    const uint4 u = a[t];
    const uint2 v = b[t];
    IdctMap m;
    m.plane = reinterpret_cast<uint8_t *>((uint64_t)u.x | (uint64_t)u.y << 32);
    m.stride = (int32_t)u.z;
    m.h_limit = (int32_t)u.w;
    m.xy = v.x;
    m.misc = v.y;
    return m;
  }
};

// Requests one tile (thread 0 only): one TMA tensor copy brings the run of blocks that starts at the tile's first
// block (always a full box of HCJ_IDCT_THREADS blocks: the rows behind the tile's own belong to the next tile or
// are filled with zeros past the end of the buffer), two small bulk copies the quant tables and the 48 bytes of
// wide-block flags; all of them complete on the stage's mbarrier.
__device__ __forceinline__ void idct_issue(const DecodeBatchDev &b, const IdctTile &t, IdctStage &st) {
  mbar_arrive_expect_tx(&st.full, IDCT_MAX_THREADS * 128u + t.qbytes + IDCT_FLAG_U4 * 16u);
  tma_tile_g2s(st.tile, b.coef_map, (int32_t)t.blk0, &st.full);
  bulk_g2s(st.q, b.qtables + t.qt_off, t.qbytes, &st.full);  // comp k uses table slot k
  bulk_g2s(st.flags, reinterpret_cast<const uint4 *>(b.wide_flags) + (t.blk0 >> 7), IDCT_FLAG_U4 * 16u, &st.full);
}

constexpr int IDCT_RING = 4;  // plan records in shared memory: tiles i .. i + 3

__device__ __forceinline__ void idct_fetch_record(const DecodeBatchDev &b, IdctTile *ring, uint32_t id, uint32_t end) {
  if (id < end) {
    cp_async16(&ring[id % IDCT_RING], &b.idct_plan[id]);
    cp_async16(reinterpret_cast<uint4 *>(&ring[id % IDCT_RING]) + 1, reinterpret_cast<const uint4 *>(&b.idct_plan[id]) + 1);
  }
  asm volatile("cp.async.commit_group;\n" ::: "memory");  // one group per call, empty past the end
}

// ------------------------------------------------------------------------------------------------
// J4: dequantise + IDCT + colour in ONE kernel for RGB24 output of 4:4:4 images (north_star: "dequantisation, 8x8
// IDCT, upsampling and YCbCr->RGB as one fused kernel"; for 4:4:4 Planar_444 is the identity).  The three blocks of an
// MCU sit in the same tile, so the samples never travel through HBM as planes:
//   1. every thread takes its block's coefficients into registers;           barrier: the staged tile is free
//   2. transform as in the planar path; the 8 x 8 samples go to an exchange area laid out as 24 rows (component,
//      row of the tile) of 8 * 42 samples inside the just-emptied stage;    barrier
//   3. the threads convert units of 8 horizontally adjacent pixels (three 8-byte reads, 24 bytes of RGB out).
// Blocks flagged for the 64-bit IDCT are transformed with the 32-bit one here like all others and put right
// afterwards by k_rgb444_fix (the rare path must not cost this one registers); images whose quant tables need the
// 64-bit path throughout are not fused (HcjImageDesc::fused_rgb is decided on the host).
// ------------------------------------------------------------------------------------------------
constexpr int FUSED_ROW_PITCH = 8 * (IDCT_MAX_THREADS / 3);  // 336 bytes: one sample row of the widest 4:4:4 tile

// YCbCr -> RGB (the stated formula, DESIGN.md 5) for one pixel, packed 0x00BBGGRR.  The -128 offsets of Cb / Cr are
// folded into the rounding constants, so a channel is one multiply-add, one shift and one add.
__device__ __forceinline__ uint32_t ycc_to_rgb_raw(int Y, int Cb, int Cr) {
  const int r = Y + ((91881 * Cr + (32768 - 91881 * 128)) >> 16);
  const int g = Y + ((-22554 * Cb - 46802 * Cr + (32768 + (22554 + 46802) * 128)) >> 16);
  const int bl = Y + ((116130 * Cb + (32768 - 116130 * 128)) >> 16);
  uint32_t t, px;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(0), "r"(bl), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(px) : "r"(g), "r"(r), "r"(t));
  return px;
}

// 4 pixels -> 12 bytes of RGB: the stated formula (DESIGN.md 5) with the "+ Y" and the rounding constant folded into the
// accumulator of the multiply-adds: Y + ((k * C + 32768) >> 16) == ((Y << 16 | 0x8000) + k * C) >> 16 exactly (the shift
// is arithmetic and Y << 16 is a multiple of 65536).  wcb_s / wcr_s: the chroma bytes with bit 7 flipped (= C - 128 as
// signed bytes); one dp4a each extracts a sign-extended sample, one PRMT builds the accumulator.
template <int I>
__device__ __forceinline__ uint32_t ycc_pixel(uint32_t wy, uint32_t wcb_s, uint32_t wcr_s) {
  const int t = (int)__byte_perm(wy, 0x00008000u, 0x4054 | (I << 8));
  // the sign-extended chroma bytes come from dp4a (x . one-hot byte selector), not from a PRMT: the colour kernels are bound
  // by the alu pipe (78 % busy against 18 % for the fma pipe), k_rgb_sub_pairs 2.39 -> 2.27 ms per 1024 x 1080p; the
  // accumulator built the same way (dp4a + IMAD for one PRMT) 2.25 ms: not kept
  const int cb = __dp4a((int)wcb_s, 1 << (8 * I), 0), cr = __dp4a((int)wcr_s, 1 << (8 * I), 0);
  const int r = (91881 * cr + t) >> 16;
  const int g = (-46802 * cr + (-22554 * cb + t)) >> 16;
  const int bl = (116130 * cb + t) >> 16;
  uint32_t u, px;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(u) : "r"(0), "r"(bl), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(px) : "r"(g), "r"(r), "r"(u));
  return px;
}
__device__ __forceinline__ void ycc4_to_rgb12(uint32_t wy, uint32_t wcb, uint32_t wcr, uint32_t *o) {
  const uint32_t sb = wcb ^ 0x80808080u, sr = wcr ^ 0x80808080u;
  const uint32_t p0 = ycc_pixel<0>(wy, sb, sr), p1 = ycc_pixel<1>(wy, sb, sr), p2 = ycc_pixel<2>(wy, sb, sr), p3 = ycc_pixel<3>(wy, sb, sr);
  o[0] = __byte_perm(p0, p1, 0x4210);  // p0 | p1 << 24
  o[1] = __byte_perm(p1, p2, 0x5421);  // p1 >> 8 | p2 << 16
  o[2] = __byte_perm(p2, p3, 0x6542);  // p2 >> 16 | p3 << 8
}
// 8 pixels -> 24 bytes of RGB
__device__ __forceinline__ void ycc8_to_rgb24(uint2 vy, const uint32_t (&cb)[2], const uint32_t (&cr)[2], uint32_t (&o)[6]) {
  ycc4_to_rgb12(vy.x, cb[0], cr[0], o);
  ycc4_to_rgb12(vy.y, cb[1], cr[1], o + 3);
}
__device__ __forceinline__ void idct_tile_rgb444(const DecodeBatchDev &b, const IdctTile &t, IdctStage &st, const IdctMap &mp, int tid) {
  uint8_t *xch = reinterpret_cast<uint8_t *>(st.tile);
  const bool mine = (mp.misc & (1u << 10)) != 0u;
  const int slot = (int)(mp.misc & 255u);
  const int c = (int)((mp.misc >> 8) & 3u);
  // (the threads beyond the tile's blocks run along on block 0 and store nothing: no conditionally defined registers
  // across the barrier, which the compiler would keep in local memory)
  uint32_t cw[32];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const uint4 u = st.tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  __syncthreads();  // every block of the tile is in registers: the stage becomes the exchange area
  {
    uint32_t pix[16];
    reconstruct_fast<false>(cw, st.q + c * 128 + 64, pix);
    uint8_t *dst = xch + c * 8 * FUSED_ROW_PITCH + (mp.xy & 0xffffu);  // x inside the tile = 8 * MCU
    if (mine) {
#pragma unroll
      for (int r = 0; r < 8; r++) *reinterpret_cast<uint2 *>(dst + r * FUSED_ROW_PITCH) = make_uint2(pix[2 * r], pix[2 * r + 1]);
    }
  }
  __syncthreads();
  const HcjImageDesc &d = b.descs[t.img];
  const int tm = t.tm, width = d.width, height = d.height;
  const int x_tile = (int)t.m0 * 8, y_tile = (int)t.my * 8;
  uint8_t *out = b.out + d.out_off;
  for (int u = tid; u < 8 * tm; u += IDCT_MAX_THREADS) {
    const int r = u / tm, m = u - r * tm;
    const int x = x_tile + m * 8, y = y_tile + r;
    if (y >= height || x >= width) continue;
    const uint2 vy = *reinterpret_cast<const uint2 *>(xch + r * FUSED_ROW_PITCH + m * 8);
    const uint2 vu = *reinterpret_cast<const uint2 *>(xch + (8 + r) * FUSED_ROW_PITCH + m * 8);
    const uint2 vv = *reinterpret_cast<const uint2 *>(xch + (16 + r) * FUSED_ROW_PITCH + m * 8);
    uint32_t o[6];
    {
      const uint32_t cb[2] = {vu.x, vu.y}, cr[2] = {vv.x, vv.y};
      ycc8_to_rgb24(vy, cb, cr, o);
    }
    uint8_t *dst = out + ((size_t)y * width + x) * 3;
    const int n = min(8, width - x);
    if (n == 8 && (reinterpret_cast<uintptr_t>(dst) & 7u) == 0) {
      reinterpret_cast<uint2 *>(dst)[0] = make_uint2(o[0], o[1]);
      reinterpret_cast<uint2 *>(dst)[1] = make_uint2(o[2], o[3]);
      reinterpret_cast<uint2 *>(dst)[2] = make_uint2(o[4], o[5]);
    } else {
      store_any<6>(dst, o, 3 * n);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// J4 for sub-sampled images (4:2:0 / 4:2:2 of even size): dequantise + IDCT + Planar_444 up-sampling + colour in the
// same kernel.  The tile's samples go to the exchange area (luma rows, then Cb rows, then Cr rows); units of 8 luma
// pixels are then converted with Planar_444's interpolation (tools/src/planar_444.ml:25-33,82-103: the chroma sample,
// its right neighbour, the row below and its right neighbour, clamped at the cropped plane's edge) done four samples
// at a time in SIMD-within-a-register form.  Two kinds of units need chroma samples of another tile - the last pixel
// row of an MCU row (the chroma row below) and the last unit of a tile's rows (the chroma column to the right): for
// those the tile writes its luma samples to the plane buffer instead, every tile writes its chroma blocks there, and
// k_rgb_deferred converts them (about 9 % of the pixels of a 1080p frame) once all tiles are done.
// Blocks flagged for the 64-bit IDCT are redone from the coefficient buffer inside the tile (wide_block_to_xch).
// ------------------------------------------------------------------------------------------------
__device__ __noinline__ void wide_block_to_xch(const int16_t *coefs_blk, const int32_t *q, uint8_t *dst, int pitch) {
  uint32_t pix[16];
  reconstruct_wide(reinterpret_cast<const uint32_t *>(coefs_blk), q, pix);
  for (int r = 0; r < 8; r++) *reinterpret_cast<uint2 *>(dst + r * pitch) = make_uint2(pix[2 * r], pix[2 * r + 1]);
}

// (a + b + 1) >> 1 of the four bytes of each word
__device__ __forceinline__ uint32_t avg2_bytes(uint32_t a, uint32_t b) { return (a | b) - (((a ^ b) >> 1) & 0x7f7f7f7fu); }
// (a + b + c + d + 2) >> 2 of the four bytes of each word, in two 16-bit lanes per word
__device__ __forceinline__ uint32_t avg4_bytes(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  const uint32_t m = 0x00ff00ffu;
  const uint32_t lo = (a & m) + (b & m) + (c & m) + (d & m) + 0x00020002u;
  const uint32_t hi = ((a >> 8) & m) + ((b >> 8) & m) + ((c >> 8) & m) + ((d >> 8) & m) + 0x00020002u;
  return ((lo >> 2) & m) | (((hi >> 2) & m) << 8);
}
// Planar_444's chroma for 8 horizontally adjacent pixels: A = the four chroma samples under them, a4 = the next one to
// the right (already clamped), B / b4 = the same of the chroma row below (or of the same row); oy: odd luma row of a
// vertically sub-sampled plane.  w[0] = pixels 0..3, w[1] = pixels 4..7.
__device__ __forceinline__ void upsample8(uint32_t A, uint32_t a4, uint32_t B, uint32_t b4, bool oy, uint32_t (&w)[2]) {
  const uint32_t A1 = (A >> 8) | (a4 << 24), B1 = (B >> 8) | (b4 << 24);
  uint32_t even, odd;
  if (!oy) {
    even = A;
    odd = avg2_bytes(A, A1);
  } else {
    even = avg2_bytes(A, B);
    odd = avg4_bytes(A, A1, B, B1);
  }
  w[0] = __byte_perm(even, odd, 0x5140);
  w[1] = __byte_perm(even, odd, 0x7362);
}
// chroma samples cx0 .. cx0 + 8 of a row (8-byte aligned), clamped at the plane's last column (nvalid = samples from
// cx0 that exist, >= 1): the eight under a unit of 16 pixels and their right neighbour
__device__ __forceinline__ void chroma9(const uint8_t *row, int nvalid, uint32_t &c0, uint32_t &c1, uint32_t &c8) {
  const uint2 v = *reinterpret_cast<const uint2 *>(row);
  c0 = v.x, c1 = v.y;
  if (nvalid >= 9) {
    c8 = *reinterpret_cast<const uint32_t *>(row + 8) & 0xffu;  // (the exchange area / the padded plane continues behind the last sample)
  } else {
    uint64_t w = (uint64_t)c0 | (uint64_t)c1 << 32;
    const uint64_t last = (w >> (8 * (nvalid - 1))) & 0xffull;
    for (int k = nvalid; k < 8; k++) w = (w & ~(0xffull << (8 * k))) | (last << (8 * k));
    c0 = (uint32_t)w, c1 = (uint32_t)(w >> 32), c8 = (uint32_t)last;
  }
}
// The chroma samples of a unit of 16 pixels: eight and their right neighbour
struct Chroma9 {
  uint32_t c0, c1, c8;
};
__device__ __forceinline__ Chroma9 load_chroma9(const uint8_t *row, int nvalid) {
  Chroma9 c;
  chroma9(row, nvalid, c.c0, c.c1, c.c8);
  return c;
}
// A unit of 16 pixels: Planar_444's up-sampling of a chroma row (and, for an odd luma row of a vertically sub-sampled
// plane, the row below) + colour conversion -> 48 bytes of RGB in o[12]
__device__ __forceinline__ void sub_unit16_convert(const uint4 vy, const Chroma9 &ba, const Chroma9 &bb, const Chroma9 &ra, const Chroma9 &rb,
                                                   bool oy, uint32_t (&o)[12]) {
  uint32_t wb[4], wr[4], w[2];
  upsample8(ba.c0, ba.c1 & 0xffu, bb.c0, bb.c1 & 0xffu, oy, w);
  wb[0] = w[0], wb[1] = w[1];
  upsample8(ba.c1, ba.c8, bb.c1, bb.c8, oy, w);
  wb[2] = w[0], wb[3] = w[1];
  upsample8(ra.c0, ra.c1 & 0xffu, rb.c0, rb.c1 & 0xffu, oy, w);
  wr[0] = w[0], wr[1] = w[1];
  upsample8(ra.c1, ra.c8, rb.c1, rb.c8, oy, w);
  wr[2] = w[0], wr[3] = w[1];
  ycc4_to_rgb12(vy.x, wb[0], wr[0], o);
  ycc4_to_rgb12(vy.y, wb[1], wr[1], o + 3);
  ycc4_to_rgb12(vy.z, wb[2], wr[2], o + 6);
  ycc4_to_rgb12(vy.w, wb[3], wr[3], o + 9);
}
__device__ __forceinline__ void sub_unit16_to_rgb(const uint4 vy, const uint8_t *cb_a, const uint8_t *cb_b, const uint8_t *cr_a,
                                                  const uint8_t *cr_b, int nvalid, bool oy, uint32_t (&o)[12]) {
  const Chroma9 ba = load_chroma9(cb_a, nvalid), ra = load_chroma9(cr_a, nvalid);
  Chroma9 bb = ba, rb = ra;
  if (oy) bb = load_chroma9(cb_b, nvalid), rb = load_chroma9(cr_b, nvalid);
  sub_unit16_convert(vy, ba, bb, ra, rb, oy, o);
}

__device__ __forceinline__ void idct_tile_rgb_sub(const DecodeBatchDev &b, const IdctTile &t, IdctStage &st, const IdctMap &mp, int tid) {
  uint8_t *xch = reinterpret_cast<uint8_t *>(st.tile);
  const bool mine = (mp.misc & (1u << 10)) != 0u;
  const int slot = (int)(mp.misc & 255u);
  const int c = (int)((mp.misc >> 8) & 3u);
  const uint32_t fbit = (uint32_t)(t.blk0 & 127u) + slot;  // bit index inside the staged flag chunks
  const bool wide = mine && ((reinterpret_cast<const uint32_t *>(st.flags)[fbit >> 5] >> (fbit & 31u)) & 1u);
  uint32_t cw[32];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const uint4 u = st.tile[slot * 8 + (j ^ (slot & 7))];
    cw[4 * j] = u.x, cw[4 * j + 1] = u.y, cw[4 * j + 2] = u.z, cw[4 * j + 3] = u.w;
  }
  const bool any_wide = __syncthreads_or(wide);  // every block of the tile is in registers: the stage becomes the exchange area
  const HcjImageDesc &d = b.descs[t.img];
  const int tm = t.tm, vs_log = d.comp[0].vs == 2 ? 1 : 0;
  const int rows = 8 << vs_log, pitch_l = 16 * tm, pitch_c = 8 * tm;
  uint8_t *xcb = xch + rows * pitch_l, *xcr = xcb + 8 * pitch_c;
  const int x = (int)t.m0 * (int)((mp.misc >> 12) & 63u) + (int)(mp.xy & 0xffffu);  // the block's place in its padded plane
  const int y = (int)t.my * (int)((mp.misc >> 18) & 63u) + (int)(mp.xy >> 16);
  uint8_t *dst = c == 0 ? xch + (mp.xy >> 16) * pitch_l + (mp.xy & 0xffffu) : (c == 1 ? xcb : xcr) + (mp.xy & 0xffffu);
  const int pitch = c == 0 ? pitch_l : pitch_c;
  {
    uint32_t pix[16];
    reconstruct_fast<false>(cw, st.q + c * 128 + 64, pix);
    if (mine && !wide) {
#pragma unroll
      for (int r = 0; r < 8; r++) *reinterpret_cast<uint2 *>(dst + r * pitch) = make_uint2(pix[2 * r], pix[2 * r + 1]);
      if (c != 0) store_block_rows(pix, mp.plane, mp.stride, x, y, mp.stride, mp.h_limit);  // for the neighbours' deferred units
    }
  }
  if (any_wide && wide) {  // rare
    const int16_t *cb = b.coefs + (t.blk0 + (uint64_t)slot) * 64;
    wide_block_to_xch(cb, st.q + c * 128, dst, pitch);
    if (c != 0) wide_block_store(reinterpret_cast<const uint32_t *>(cb), st.q + c * 128, mp.plane, mp.stride, x, y, mp.stride, mp.h_limit);
  }
  __syncthreads();
  const int width = d.width, height = d.height, cwid = d.comp[1].actual_w, chh = d.comp[1].actual_h;
  const int x_tile = (int)t.m0 * 16, y_tile = (int)t.my * rows, cx_tile = (int)t.m0 * 8, cy_tile = (int)t.my * 8;
  const bool right_deferred = cx_tile + 8 * tm < cwid;           // the chroma column right of the tile exists
  const bool bottom_deferred = vs_log && cy_tile + 8 < chh;      // the chroma row below the tile exists
  uint8_t *out = b.out + d.out_off;
  uint8_t *plane_y = b.planes + d.comp[0].plane_off;
  const int stride_y = d.comp[0].decoded_w;
  // Units of 16 pixels (one MCU column of one pixel row), all even rows first, then all odd rows: the lanes of a warp
  // run the same interpolation code.
  const int nunits = rows * tm, nhalf = vs_log ? 8 * tm : nunits;
  const uint32_t recip = 65536u / (uint32_t)tm + 1u;  // k / tm for k < 2^11, tm <= 32
  for (int idx = tid; idx < nunits; idx += IDCT_MAX_THREADS) {
    const int k = idx < nhalf ? idx : idx - nhalf;
    const int rk = (int)(((uint32_t)k * recip) >> 16), m = k - rk * tm;
    const int r = vs_log ? 2 * rk + (idx < nhalf ? 0 : 1) : rk;
    const int px = x_tile + 16 * m, py = y_tile + r;
    if (py >= height || px >= width) continue;
    const uint4 vy = *reinterpret_cast<const uint4 *>(xch + r * pitch_l + 16 * m);
    if ((right_deferred && m == tm - 1) || (bottom_deferred && r == rows - 1)) {
      *reinterpret_cast<uint4 *>(plane_y + (size_t)py * stride_y + px) = vy;  // k_rgb_deferred converts the group
      continue;
    }
    const int crow = r >> vs_log;
    const bool oy = vs_log && (r & 1);
    // the row below, clamped at the cropped plane's last row (inside the tile here: the other case is deferred)
    const int crow1 = (oy && cy_tile + crow + 1 <= chh - 1) ? crow + 1 : crow;
    const int nvalid = cwid - (cx_tile + 8 * m);
    uint32_t o[12];
    sub_unit16_to_rgb(vy, xcb + crow * pitch_c + 8 * m, xcb + crow1 * pitch_c + 8 * m, xcr + crow * pitch_c + 8 * m,
                      xcr + crow1 * pitch_c + 8 * m, nvalid, oy, o);
    store_any<12>(out + ((size_t)py * width + px) * 3, o, 3 * min(16, width - px));
  }
}

// FUSED = true is the instance launched for RGB24 batches that hold 4:4:4 images: their tiles take the fused path
// (idct_tile_rgb444 below); every other tile, and every tile of the FUSED = false instance, takes the planar path.
// K: samples per block side in the output planes; K = 4, 2, 1 are the scaled decodes (HCJ_FLAG_SCALE_*, never fused),
// which keep the tile plan, the staging and the thread -> block mapping and change only the transform and the store.
// ISLOW (K = 8, never fused) is the libjpeg reconstruction (HCJ_FLAG_LIBJPEG) in the same frame.
template <bool FUSED, int K = 8, bool ISLOW = false>
__global__ void __launch_bounds__(IDCT_MAX_THREADS, HCJ_IDCT_CTAS_PER_SM)
    k_idct_persistent(const __grid_constant__ DecodeBatchDev b, int mode) {
  extern __shared__ uint4 s_dyn[];
  // 1 KiB alignment for the swizzled tiles (the launch asks for 1 KiB more than two stages)
  IdctStage *stages = reinterpret_cast<IdctStage *>(reinterpret_cast<uint8_t *>(s_dyn) + ((1024u - (smem_u32(s_dyn) & 1023u)) & 1023u));
  const int tid = threadIdx.x;
  const uint32_t total = b.tile_hi - b.tile_lo;
  const uint32_t chunk = (total + gridDim.x - 1) / gridDim.x;
  const uint32_t begin = b.tile_lo + min(blockIdx.x * chunk, total), end = b.tile_lo + min((blockIdx.x + 1) * chunk, total);
  if (begin >= end) return;

  __shared__ IdctTile s_ring[IDCT_RING];  // record of tile id at s_ring[id % IDCT_RING]
  __shared__ IdctMapSmem s_map;
  if (tid == 0) {
    mbar_init(&stages[0].full, 1);
    mbar_init(&stages[1].full, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    idct_fetch_record(b, s_ring, begin, end);
    idct_fetch_record(b, s_ring, begin + 1, end);
    idct_fetch_record(b, s_ring, begin + 2, end);
    asm volatile("cp.async.wait_group 1;\n" ::: "memory");  // records of begin and begin + 1 are in
    idct_issue(b, s_ring[begin % IDCT_RING], stages[0]);
  }
  __syncthreads();
  for (uint32_t id = begin; id < end; id++) {
    const int buf = (int)(id - begin) & 1;
    IdctStage &st = stages[buf];
    if (tid == 0) {
      // the record of id + 1 arrived before the previous barrier; ask for id + 3, whose slot held id - 1
      idct_fetch_record(b, s_ring, id + 3, end);
      if (id + 1 < end) idct_issue(b, s_ring[(id + 1) % IDCT_RING], stages[buf ^ 1]);
    }
    const IdctTile &t = s_ring[id % IDCT_RING];
    if (t.remap || id == begin) {  // CTA-uniform: new image or a narrower last tile in the row; only this thread reads its entry
      const HcjImageDesc &d = b.descs[t.img];
      const int tm = t.tm;
      int rem = tid, c = 0;
      for (; c < d.ncomp - 1; c++) {
        int n = tm * d.comp[c].hs * d.comp[c].vs;
        if (rem < n) break;
        rem -= n;
      }
      const HcjCompGeom &g = d.comp[c];
      const int rowlen = tm * g.hs;
      const int by = (rem >= rowlen) + (rem >= 2 * rowlen) + (rem >= 3 * rowlen);  // vs <= 4
      const int r2 = rem - by * rowlen;
      const int m = g.hs == 1 ? r2 : g.hs == 2 ? r2 >> 1 : g.hs == 4 ? r2 >> 2 : r2 / 3;
      const int bx = r2 - m * g.hs;
      const uint32_t slot = (uint32_t)(m * d.bpm + g.first_blk + by * g.hs + bx);
      const bool mine = tid < (int)t.nblk;
      IdctMap mp;
      mp.xy = (uint32_t)(m * g.hs * K + bx * K) | (uint32_t)(by * K) << 16;
      mp.misc = (mine ? slot : 0u) | (uint32_t)c << 8 | (mine ? 1u << 10 : 0u) | (d.wide_idct ? 1u << 11 : 0u) |
                (uint32_t)(g.hs * K) << 12 | (uint32_t)(g.vs * K) << 18;
      if (mode == 0) {
        mp.plane = b.out + d.out_off + g.out_off;
        mp.stride = g.actual_w;
        mp.h_limit = g.actual_h;
      } else {
        mp.plane = (mode == 2 ? b.planes : b.out + d.out_off) + g.plane_off;
        mp.stride = g.decoded_w;
        mp.h_limit = g.decoded_h;
      }
      s_map.put(tid, mp);
    }
    mbar_wait(&st.full, (uint32_t)((id - begin) >> 1) & 1u);  // the stage's ((id - begin) / 2)-th use
    // the thread index is read from its special register again here: kept live across the loop it ends up in a
    // local-memory spill slot, and the reload sat in front of every tile (2.25 -> 2.20 ms).  (Moving the loop counter
    // and the block's output position out of the transform's live range the same way made it slower: 2.36 ms.)
    int tnow;
    asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tnow));
    const IdctMap mp = s_map.get(tnow);
    if (FUSED && t.fused == 1u) {  // CTA-uniform
      idct_tile_rgb444(b, t, st, mp, tnow);
    } else if (FUSED && t.fused == 2u) {
      idct_tile_rgb_sub(b, t, st, mp, tnow);
    } else if ((K != 8 || ISLOW) && (mp.misc & (1u << 10))) {
      const int slot = (int)(mp.misc & 255u);
      const uint32_t fbit = (uint32_t)(t.blk0 & 127u) + slot;
      const bool wide = (mp.misc & (1u << 11)) || ((reinterpret_cast<const uint32_t *>(st.flags)[fbit >> 5] >> (fbit & 31u)) & 1u);
      const int x = (int)t.m0 * (int)((mp.misc >> 12) & 63u) + (int)(mp.xy & 0xffffu);
      const int y = (int)t.my * (int)((mp.misc >> 18) & 63u) + (int)(mp.xy >> 16);
      if (ISLOW) islow_block_store(st.tile, slot, st.q + ((mp.misc >> 8) & 3u) * 128u, wide, mp.plane, mp.stride, x, y, mp.h_limit);
      else scaled_block_store<K>(st.tile, slot, st.q + ((mp.misc >> 8) & 3u) * 128u, wide, mp.plane, mp.stride, x, y, mp.h_limit);
    } else if (K == 8 && (mp.misc & (1u << 10))) {
      const int slot = (int)(mp.misc & 255u);
      uint32_t cw[32];
#pragma unroll
      for (int j = 0; j < 8; j++) {
        uint4 u = st.tile[slot * 8 + (j ^ (slot & 7))];
        cw[4 * j] = u.x;
        cw[4 * j + 1] = u.y;
        cw[4 * j + 2] = u.z;
        cw[4 * j + 3] = u.w;
      }
      const uint32_t fbit = (uint32_t)(t.blk0 & 127u) + slot;  // bit index inside the staged flag chunks
      const bool wide = (mp.misc & (1u << 11)) || ((reinterpret_cast<const uint32_t *>(st.flags)[fbit >> 5] >> (fbit & 31u)) & 1u);
      const int x = (int)t.m0 * (int)((mp.misc >> 12) & 63u) + (int)(mp.xy & 0xffffu);
      const int y = (int)t.my * (int)((mp.misc >> 18) & 63u) + (int)(mp.xy >> 16);
      const int32_t *q = st.q + ((mp.misc >> 8) & 3u) * 128u;
      if (wide) {
        wide_block_store_staged(st.tile, slot, q, mp.plane, mp.stride, x, y, mp.stride, mp.h_limit);
      } else {
        uint32_t pix[16];
        reconstruct_fast<false>(cw, q + 64, pix);
        store_block_rows(pix, mp.plane, mp.stride, x, y, mp.stride, mp.h_limit);
      }
    }
    if (tid == 0) asm volatile("cp.async.wait_group 1;\n" ::: "memory");  // the record of id + 2 is in (id + 3 may be in flight)
    __syncthreads();  // this stage is refilled by the next iteration's prefetch; the ring slot of id by the next fetch
  }
}

constexpr size_t IDCT_SMEM = 2 * sizeof(IdctStage) + 1024;

void launch_idct(const DecodeBatchDev &b, int mode, cudaStream_t s) {
  if (b.img_hi <= b.img_lo || b.tile_hi <= b.tile_lo) return;
  const int grid = HCJ_IDCT_CTAS_PER_SM * (b.sm_count > 0 ? b.sm_count : 148);
  k_idct_plan<<<dim3((b.max_idct_tiles + 127) / 128, b.img_hi - b.img_lo), 128, 0, s>>>(b);
  const uint32_t total = b.tile_hi - b.tile_lo;
  const unsigned ctas = (unsigned)(total < (uint32_t)grid ? total : grid);
  if (b.islow) k_idct_persistent<false, 8, true><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
  else if (b.block_k == 4) k_idct_persistent<false, 4><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
  else if (b.block_k == 2) k_idct_persistent<false, 2><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
  else if (b.block_k == 1) k_idct_persistent<false, 1><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
  else if (mode == 2 && (b.has_fused || b.has_fused_sub)) k_idct_persistent<true><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
  else k_idct_persistent<false><<<ctas, IDCT_MAX_THREADS, IDCT_SMEM, s>>>(b, mode);
}

// The coefficient buffer as the TMA unit sees it: uint16 [total blocks][64], box = HCJ_IDCT_THREADS blocks x 64,
// 128-byte swizzle, zeros out of bounds.  cuTensorMapEncodeTiled is looked up through the runtime (no -lcuda).
int make_coef_tensor_map(DecodeBatchDev *b) {
  typedef CUresult (*EncodeTiled)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeTiled encode = nullptr;
  if (!encode) {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess) return (int)e;
    if (q != cudaDriverEntryPointSuccess || !fn) return (int)cudaErrorNotSupported;
    encode = reinterpret_cast<EncodeTiled>(fn);
  }
  static_assert(sizeof(CUtensorMap) == sizeof(b->coef_map), "CUtensorMap is 128 bytes");
  const cuuint64_t dims[2] = {64, b->total_blocks ? b->total_blocks : 1};
  const cuuint64_t strides[1] = {128};  // bytes from one block to the next
  const cuuint32_t box[2] = {64, IDCT_MAX_THREADS};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = encode(reinterpret_cast<CUtensorMap *>(b->coef_map), CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, b->coefs, dims, strides, box,
                      estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

// Debug tap: Component.recon of caller-provided blocks (hcj_idct_blocks).
__global__ void k_idct_blocks(const int16_t *coefs, size_t nblocks, const uint16_t *qt, int force_wide, uint8_t *out) {
  __shared__ int32_t s_q[128];
  if (threadIdx.x < 64) {
    s_q[threadIdx.x] = qt[threadIdx.x];
    s_q[64 + threadIdx.x] = HCJ_QD(threadIdx.x, qt[threadIdx.x]);
  }
  __syncthreads();
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nblocks) return;
  uint32_t cw[32], pix[16];
  const uint4 *src = reinterpret_cast<const uint4 *>(coefs + i * 64);
#pragma unroll
  for (int j = 0; j < 8; j++) {
    uint4 u = __ldg(src + j);
    cw[4 * j] = u.x;
    cw[4 * j + 1] = u.y;
    cw[4 * j + 2] = u.z;
    cw[4 * j + 3] = u.w;
  }
  if (force_wide || !reconstruct_fast<true>(cw, s_q + 64, pix)) {
    wide_block_store(reinterpret_cast<const uint32_t *>(coefs + i * 64), s_q, out + i * 64, 8, 0, 0, 8, 8);
    return;
  }
  uint4 *dst = reinterpret_cast<uint4 *>(out + i * 64);
#pragma unroll
  for (int j = 0; j < 4; j++) dst[j] = make_uint4(pix[4 * j], pix[4 * j + 1], pix[4 * j + 2], pix[4 * j + 3]);
}

void launch_idct_blocks(const int16_t *coefs, size_t nblocks, const uint16_t *qt, bool force_wide, uint8_t *out,
                        cudaStream_t s) {
  if (nblocks == 0) return;
  k_idct_blocks<<<(unsigned)((nblocks + 127) / 128), 128, 0, s>>>(coefs, nblocks, qt, force_wide ? 1 : 0, out);
}

// ================================================================================================
// K9: Planar_444 up-sampling (tools/src/planar_444.ml:25-33,82-103) + YCbCr -> RGB24 (stated formula,
// DESIGN.md: JFIF full range, 16-bit fixed point).  One thread per 4 horizontally adjacent pixels.
// Reads the padded planes written by k_idct_persistent (mode 2); the up-sampling clamps at the CROPPED plane
// edge, as Planar_444 does on the cropped frame.
// ================================================================================================
__device__ __forceinline__ int up_sample(const uint8_t *p, int stride, int w, int h, int x, int y, int hs_log, int vs_log) {
  // hs_log / vs_log: 1 if this axis is subsampled by 2.  (x, y) in full-resolution coordinates.
  int cx = x >> hs_log, cy = y >> vs_log;
  // odd luma sizes: Planar_444 never writes the last column / row of the (zero-initialised) 4:4:4 plane
  if (cx >= w || cy >= h) return 0;
  int cx1 = min(cx + 1, w - 1), cy1 = min(cy + 1, h - 1);
  int a = p[cy * stride + cx];
  bool ox = hs_log && (x & 1), oy = vs_log && (y & 1);
  if (!ox && !oy) return a;
  if (ox && !oy) return (a + p[cy * stride + cx1] + 1) >> 1;
  if (!ox && oy) return (a + p[cy1 * stride + cx] + 1) >> 1;
  // the model's edge columns use avg2 of the two rows (planar_444.ml:97-102); with cx1 == cx that is
  // what avg4(a, a, c, c) would NOT give after rounding, so treat the edge explicitly
  if (cx1 == cx) return (a + p[cy1 * stride + cx] + 1) >> 1;
  return (a + p[cy * stride + cx1] + p[cy1 * stride + cx] + p[cy1 * stride + cx1] + 2) >> 2;
}

// The stated colour formula (DESIGN.md §5) for one pixel, packed 0x00BBGGRR.
__device__ __forceinline__ uint32_t ycc_to_rgb(int Y, int Cb, int Cr) {
  Cb -= 128;
  Cr -= 128;
  const int r = Y + ((91881 * Cr + 32768) >> 16);
  const int g = Y + ((-22554 * Cb - 46802 * Cr + 32768) >> 16);
  const int bl = Y + ((116130 * Cb + 32768) >> 16);
  // clamp to [0, 255] and pack: two saturating packs instead of six min / max and the shifts
  uint32_t t, px;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(0), "r"(bl), "r"(0));
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(px) : "r"(g), "r"(r), "r"(t));
  return px;
}

// 16 bytes from an 8-byte aligned address
__device__ __forceinline__ void load16(const uint8_t *p, uint32_t (&w)[4]) {
  if ((reinterpret_cast<uintptr_t>(p) & 15u) == 0) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
    w[0] = v.x, w[1] = v.y, w[2] = v.z, w[3] = v.w;
  } else {
    const uint2 a = __ldg(reinterpret_cast<const uint2 *>(p)), c = __ldg(reinterpret_cast<const uint2 *>(p) + 1);
    w[0] = a.x, w[1] = a.y, w[2] = c.x, w[3] = c.y;
  }
}

// The sub-sampled group of k_rgb.  EDGE: the group is the short last one of its row (or touches the odd last column):
// only then are neighbours replicated inside the group and samples past the chroma plane zeroed.  Returns true if
// it has stored the pixels (RGB24), false if the caller stores the planar words.
template <bool PLANAR, bool EDGE>
__device__ __forceinline__ bool rgb_sub_group(const DecodeBatchDev &b, const HcjImageDesc &d, const uint8_t *pu, const uint8_t *pv, int su,
                                              int sv, int cw, int chh, int vs_log, int x0, int y, int n, const uint32_t (&wy)[4],
                                              uint32_t (&wu)[4], uint32_t (&wv)[4]) {
  const int cy = y >> vs_log, cx0 = x0 >> 1;
  const bool oy = vs_log && (y & 1);
  if (!PLANAR && (d.width & 1) == 0 && (!vs_log || (d.height & 1) == 0)) {
    // even sizes (every luma sample has its chroma sample): interpolation and colour four samples at a time
    const int cy1 = oy ? min(cy + 1, chh - 1) : cy;
    uint32_t o[12];
    sub_unit16_to_rgb(make_uint4(wy[0], wy[1], wy[2], wy[3]), pu + (size_t)cy * su + cx0, pu + (size_t)cy1 * su + cx0,
                      pv + (size_t)cy * sv + cx0, pv + (size_t)cy1 * sv + cx0, cw - cx0, oy, o);
    store_any<12>(b.out + d.out_off + ((size_t)y * d.width + x0) * 3, o, 3 * n);
    return true;
  }
  const bool below = cy >= chh;  // odd height: no chroma row for the last luma row
  const int cy1 = min(cy + 1, chh - 1), cx8 = max(min(cx0 + 8, cw - 1), 0);
  int cu[2][9], cv[2][9];
#pragma unroll
  for (int r = 0; r < 2; r++) {
    const int row = r ? cy1 : cy;
    uint2 a = make_uint2(0u, 0u), c = make_uint2(0u, 0u);
    int a8 = 0, c8 = 0;
    if (!below && (r == 0 || oy)) {
      a = __ldg(reinterpret_cast<const uint2 *>(pu + (size_t)row * su + cx0));
      c = __ldg(reinterpret_cast<const uint2 *>(pv + (size_t)row * sv + cx0));
      a8 = __ldg(pu + (size_t)row * su + cx8);
      c8 = __ldg(pv + (size_t)row * sv + cx8);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
      cu[r][k] = (int)(((k < 4 ? a.x : a.y) >> (8 * (k & 3))) & 0xffu);
      cv[r][k] = (int)(((k < 4 ? c.x : c.y) >> (8 * (k & 3))) & 0xffu);
    }
    cu[r][8] = a8;
    cv[r][8] = c8;
    if (EDGE)
#pragma unroll
      for (int k = 1; k < 8; k++)  // a short last group: the neighbour to the right of the last sample is that sample
        if (cx0 + k > cw - 1) cu[r][k] = cu[r][k - 1], cv[r][k] = cv[r][k - 1];
  }
  uint32_t o[12];
#pragma unroll
  for (int k = 0; k < 4; k++) {  // 4 pixels -> 12 bytes = 3 words
    uint32_t px[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const int i = 4 * k + j, cpos = i >> 1;
      int Cb, Cr;
      if (!oy) {
        Cb = (i & 1) ? (cu[0][cpos] + cu[0][cpos + 1] + 1) >> 1 : cu[0][cpos];
        Cr = (i & 1) ? (cv[0][cpos] + cv[0][cpos + 1] + 1) >> 1 : cv[0][cpos];
      } else {
        Cb = (i & 1) ? (cu[0][cpos] + cu[0][cpos + 1] + cu[1][cpos] + cu[1][cpos + 1] + 2) >> 2 : (cu[0][cpos] + cu[1][cpos] + 1) >> 1;
        Cr = (i & 1) ? (cv[0][cpos] + cv[0][cpos + 1] + cv[1][cpos] + cv[1][cpos + 1] + 2) >> 2 : (cv[0][cpos] + cv[1][cpos] + 1) >> 1;
      }
      if (EDGE && cx0 + cpos >= cw) Cb = Cr = 0;  // odd width: the last luma column has no chroma sample
      if (PLANAR) {
        wu[k] |= (uint32_t)Cb << (8 * j);
        wv[k] |= (uint32_t)Cr << (8 * j);
      } else {
        px[j] = ycc_to_rgb((wy[k] >> (8 * j)) & 0xff, Cb, Cr);  // straight from the interpolated values
      }
    }
    if (!PLANAR) {
      o[3 * k + 0] = px[0] | (px[1] << 24);
      o[3 * k + 1] = (px[1] >> 8) | (px[2] << 16);
      o[3 * k + 2] = (px[2] >> 16) | (px[3] << 8);
    }
  }
  if (!PLANAR) {
    store_any<12>(b.out + d.out_off + ((size_t)y * d.width + x0) * 3, o, 3 * n);
    return true;
  }
  return false;
}

// Each thread converts 16 horizontally adjacent pixels (x0 a multiple of 16; the last group of a row may be short) in
// registers: 16 bytes per plane for 4:4:4; for 4:2:0 / 4:2:2 the 16 luma samples plus the 9 chroma samples (of one or
// two rows) they need, with Planar_444's interpolation on those - the neighbours clamped at the cropped plane's
// edge, where avg2 (a, a) = a and avg4 (a, a, c, c) = avg2 (a, c) are the model's edge cases; past the last chroma
// row / column of an odd-sized image the 4:4:4 plane is still zero.  The padded planes keep every row 8-byte
// aligned, so the loads are always vector loads; the stores adapt to the alignment of the output row (store_any).
// Two instances per output format, one for 4:4:4 images and one for sub-sampled ones (SUB), each skipping the other's
// images: the 4:4:4 path needs far fewer registers, and a batch is normally of one kind (launch_rgb starts only
// the instances the batch needs).  (Planes that are not 8-byte aligned - never produced by the library - go pixel by
// pixel through up_sample.)
template <bool PLANAR, bool SUB>  // PLANAR: planar 4:4:4 Y,U,V (Planar_444.convert_from_420 / _422 of the frame) instead of RGB24
__device__ __forceinline__ void rgb_group(const DecodeBatchDev &b, const HcjImageDesc &d, int x0, int y) {
  const uint8_t *py = b.planes + d.comp[0].plane_off, *pu = b.planes + d.comp[1].plane_off,
                *pv = b.planes + d.comp[2].plane_off;
  const int sy = d.comp[0].decoded_w, su = d.comp[1].decoded_w, sv = d.comp[2].decoded_w;
  const int hs_log = d.chroma == 444 ? 0 : 1, vs_log = d.chroma == 420 ? 1 : 0;
  const int cw = d.comp[1].actual_w, chh = d.comp[1].actual_h;
  const int n = min(16, d.width - x0);  // pixels of this group
  const bool aligned8 = ((sy | su | sv) & 7) == 0 && (((uintptr_t)py | (uintptr_t)pu | (uintptr_t)pv) & 7u) == 0 &&
                        d.comp[2].actual_w == cw && d.comp[2].actual_h == chh;
  uint32_t wy[4], wu[4] = {0u, 0u, 0u, 0u}, wv[4] = {0u, 0u, 0u, 0u};
  if (aligned8 && (!SUB ? !hs_log : (hs_log && su * 2 >= sy && sv * 2 >= sy))) {
    load16(py + (size_t)y * sy + x0, wy);
    if (!SUB) {
      load16(pu + (size_t)y * su + x0, wu);
      load16(pv + (size_t)y * sv + x0, wv);
    } else {
      const bool edge = n < 16 || ((x0 + 15) >> 1) > cw - 1;
      if (edge ? rgb_sub_group<PLANAR, true>(b, d, pu, pv, su, sv, cw, chh, vs_log, x0, y, n, wy, wu, wv)
               : rgb_sub_group<PLANAR, false>(b, d, pu, pv, su, sv, cw, chh, vs_log, x0, y, n, wy, wu, wv))
        return;
    }
    if (PLANAR) {
      const size_t plane = (size_t)d.width * d.height;
      uint8_t *oy = b.out + d.out_off + (size_t)y * d.width + x0;
      store_any<4>(oy, wy, n);
      store_any<4>(oy + plane, wu, n);
      store_any<4>(oy + 2 * plane, wv, n);
      return;
    }
    uint32_t o[12];
#pragma unroll
    for (int k = 0; k < 4; k++) {  // 4 pixels -> 12 bytes = 3 words
      uint32_t px[4];
#pragma unroll
      for (int i = 0; i < 4; i++)
        px[i] = ycc_to_rgb((wy[k] >> (8 * i)) & 0xff, (wu[k] >> (8 * i)) & 0xff, (wv[k] >> (8 * i)) & 0xff);
      o[3 * k + 0] = px[0] | (px[1] << 24);
      o[3 * k + 1] = (px[1] >> 8) | (px[2] << 16);
      o[3 * k + 2] = (px[2] >> 16) | (px[3] << 8);
    }
    store_any<12>(b.out + d.out_off + ((size_t)y * d.width + x0) * 3, o, 3 * n);
    return;
  }
  if (PLANAR) {
    const size_t plane = (size_t)d.width * d.height;
    uint8_t *oy = b.out + d.out_off + (size_t)y * d.width + x0, *ou = oy + plane, *ov = ou + plane;
    for (int i = 0; i < n; i++) {
      const int x = x0 + i;
      oy[i] = py[(size_t)y * sy + x];
      ou[i] = (uint8_t)up_sample(pu, su, cw, chh, x, y, hs_log, vs_log);
      ov[i] = (uint8_t)up_sample(pv, sv, d.comp[2].actual_w, d.comp[2].actual_h, x, y, hs_log, vs_log);
    }
    return;
  }
  uint8_t *dst = b.out + d.out_off + ((size_t)y * d.width + x0) * 3;
  for (int i = 0; i < n; i++) {
    const int x = x0 + i;
    const int Y = py[(size_t)y * sy + x];
    const int Cb = up_sample(pu, su, cw, chh, x, y, hs_log, vs_log);
    const int Cr = up_sample(pv, sv, d.comp[2].actual_w, d.comp[2].actual_h, x, y, hs_log, vs_log);
    const uint32_t px = ycc_to_rgb(Y, Cb, Cr);
    dst[3 * i + 0] = (uint8_t)px;
    dst[3 * i + 1] = (uint8_t)(px >> 8);
    dst[3 * i + 2] = (uint8_t)(px >> 16);
  }
}

template <bool PLANAR, bool SUB>
__global__ void __launch_bounds__(128, SUB ? 10 : 12) k_rgb(DecodeBatchDev b) {
  const HcjImageDesc &d = b.descs[blockIdx.z + b.img_lo];
  if (!d.valid || d.chroma == 0 || (d.chroma != 444) != SUB || (!PLANAR && d.fused_rgb)) return;
  if (!PLANAR && SUB && !(d.width & 1) && !(d.chroma == 420 && (d.height & 1))) return;  // k_rgb_sub_pairs
  const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16, y = blockIdx.y;
  if (y >= d.height || x0 >= d.width) return;
  rgb_group<PLANAR, SUB>(b, d, x0, y);
}

// RGB24 of sub-sampled images of even size, two pixel rows (2 * blockIdx.y and the next) of a 16-pixel column per thread:
// everything the pair needs - 32 luma samples, two chroma rows of nine samples per component - is requested before
// anything is computed (the one-row form of k_rgb is bound by the latency of its loads: 49 % of the HBM peak), and for
// 4:2:0 the two rows share their chroma rows.
__global__ void __launch_bounds__(128, 8) k_rgb_sub_pairs(DecodeBatchDev b) {
  const HcjImageDesc &d = b.descs[blockIdx.z + b.img_lo];
  if (!d.valid || d.chroma == 0 || d.chroma == 444 || d.fused_rgb) return;
  const int vs_log = d.chroma == 420 ? 1 : 0;
  if ((d.width & 1) || (vs_log && (d.height & 1))) return;  // odd sizes: k_rgb
  const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16, y0 = blockIdx.y * 2;
  if (y0 >= d.height || x0 >= d.width) return;
  const uint8_t *py = b.planes + d.comp[0].plane_off, *pu = b.planes + d.comp[1].plane_off, *pv = b.planes + d.comp[2].plane_off;
  const int sy = d.comp[0].decoded_w, su = d.comp[1].decoded_w, sv = d.comp[2].decoded_w;
  const int cw = d.comp[1].actual_w, chh = d.comp[1].actual_h;
  const bool two = y0 + 1 < d.height;
  const int cx0 = x0 >> 1, nvalid = cw - cx0;
  // chroma rows of the first and of the second pixel row (4:2:0: the same row, and the clamped row below it)
  const int ca = vs_log ? blockIdx.y : y0, cb_ = vs_log ? min((int)blockIdx.y + 1, chh - 1) : min(y0 + 1, chh - 1);
  uint32_t w0[4], w1[4] = {0u, 0u, 0u, 0u};
  load16(py + (size_t)y0 * sy + x0, w0);
  if (two) load16(py + (size_t)(y0 + 1) * sy + x0, w1);
  const Chroma9 ua = load_chroma9(pu + (size_t)ca * su + cx0, nvalid), va = load_chroma9(pv + (size_t)ca * sv + cx0, nvalid);
  const Chroma9 ub = load_chroma9(pu + (size_t)cb_ * su + cx0, nvalid), vb = load_chroma9(pv + (size_t)cb_ * sv + cx0, nvalid);
  const int n = min(16, d.width - x0);
  uint8_t *dst = b.out + d.out_off + ((size_t)y0 * d.width + x0) * 3;
  uint32_t o[12];
  sub_unit16_convert(make_uint4(w0[0], w0[1], w0[2], w0[3]), ua, ua, va, va, false, o);
  store_any<12>(dst, o, 3 * n);
  if (two) {
    if (vs_log) sub_unit16_convert(make_uint4(w1[0], w1[1], w1[2], w1[3]), ua, ub, va, vb, true, o);
    else sub_unit16_convert(make_uint4(w1[0], w1[1], w1[2], w1[3]), ub, ub, vb, vb, false, o);
    store_any<12>(dst + (size_t)d.width * 3, o, 3 * n);
  }
}

// The units that the fused tiles of sub-sampled images (idct_tile_rgb_sub) left over: the last pixel row of every MCU
// row that has a chroma row below it, and the last 16 pixels of the rows of every tile that has a tile to its right.
// One thread per group of 16 pixels, converted from the plane buffer like everything else in k_rgb.
// grid (ceil(max groups of an image / 128), images)
__global__ void __launch_bounds__(128, 10) k_rgb_deferred(DecodeBatchDev b) {
  const HcjImageDesc &d = b.descs[blockIdx.y + b.img_lo];
  if (!d.valid || d.fused_rgb != 2) return;
  const int vs_log = d.comp[0].vs == 2 ? 1 : 0, rows = 8 << vs_log;
  const int chh = d.comp[1].actual_h;
  const int ngroups = (d.width + 15) / 16;
  const int def_rows = vs_log ? (chh - 1) / 8 : 0;  // MCU rows my with a chroma row 8 * my + 8 below them
  int tpr;
  const int tm_bal = idct_tile_width(b, d, tpr);
  const int id = blockIdx.x * blockDim.x + threadIdx.x;
  int x0, y;
  if (id < def_rows * ngroups) {
    const int k = id / ngroups;
    x0 = (id - k * ngroups) * 16;
    y = rows * k + rows - 1;
  } else {
    const int id2 = id - def_rows * ngroups;
    const int tx = id2 / d.height;
    if (tx >= tpr - 1) return;
    y = id2 - tx * d.height;
    x0 = 16 * tm_bal * (tx + 1) - 16;
  }
  if (y >= d.height || x0 >= d.width) return;
  rgb_group<false, true>(b, d, x0, y);
}

// Fused RGB24 images: the 8 x 8 pixels of every MCU that holds a block flagged for the 64-bit IDCT (pathological
// coefficient sums, see HCJ_IDCT_L1_LIMIT) are recomputed with the model's arithmetic verbatim.  One thread per 32
// blocks of an image looks at their flags; almost all of them find nothing.  grid (ceil(max blocks / 32 / 128), images)
__global__ void __launch_bounds__(128) k_rgb444_fix(DecodeBatchDev b) {
  const HcjImageDesc &d = b.descs[blockIdx.y + b.img_lo];
  if (!d.valid || d.fused_rgb != 1) return;
  const uint32_t first = (blockIdx.x * blockDim.x + threadIdx.x) * 32u;
  if (first >= d.nblocks) return;
  const uint64_t g0 = d.coef_off + first;
  const uint32_t w0 = b.wide_flags[g0 >> 5], w1 = b.wide_flags[(g0 >> 5) + 1];
  uint32_t bits = __funnelshift_r(w0, w1, (uint32_t)(g0 & 31u));
  if (first + 32u > d.nblocks) bits &= (1u << (d.nblocks - first)) - 1u;
  uint32_t done_mcu = 0xffffffffu;
  while (bits) {
    const uint32_t blk = first + (uint32_t)__ffs((int)bits) - 1u;
    bits &= bits - 1u;
    const uint32_t mcu = blk / 3u;
    if (mcu == done_mcu) continue;
    done_mcu = mcu;
    uint32_t pix[3][16];
    for (int c = 0; c < 3; c++)
      reconstruct_wide(reinterpret_cast<const uint32_t *>(b.coefs + (d.coef_off + (uint64_t)mcu * 3u + c) * 64), b.qtables + d.qt_off + c * 128, pix[c]);
    const int x0 = (int)(mcu % (uint32_t)d.mcus_wide) * 8, y0 = (int)(mcu / (uint32_t)d.mcus_wide) * 8;
    for (int r = 0; r < 8 && y0 + r < d.height; r++)
      for (int i = 0; i < 8 && x0 + i < d.width; i++) {
        const int w = 2 * r + (i >> 2), sh = 8 * (i & 3);
        const uint32_t px = ycc_to_rgb((int)((pix[0][w] >> sh) & 0xffu), (int)((pix[1][w] >> sh) & 0xffu), (int)((pix[2][w] >> sh) & 0xffu));
        uint8_t *dst = b.out + d.out_off + ((size_t)(y0 + r) * d.width + x0 + i) * 3;
        dst[0] = (uint8_t)px, dst[1] = (uint8_t)(px >> 8), dst[2] = (uint8_t)(px >> 16);
      }
  }
}

// ================================================================================================
// K9 for HCJ_FLAG_LIBJPEG: libjpeg's up-sampling (jdsample.c, libjpeg_upsample in hcj_device.cuh) + the colour formula,
// for the images that are not 4:4:4 (those take k_rgb: libjpeg's copy is Planar_444's).  One thread per 16 horizontally
// adjacent pixels of a row.  The common layouts - luma at full size, both chroma components at ratio (2, 1) or (2, 2),
// real chroma planes wider than 2 - take the fast path: 16 luma samples and, per chroma component, 8 samples with their
// left and right neighbours from one row (h2v1) or from the near and the far row (h2v2), all requested before anything
// is computed.  Only the group at the right end of the real chroma plane (EDGE) replicates its last sample inside the
// group.  Everything else (4:4:0, 4:1:1, other layouts, planes of width <= 2) goes sample by sample.
// ================================================================================================
struct ChromaRow10 {
  uint2 m;   // samples j0 .. j0 + 7
  int l, r;  // samples j0 - 1 and j0 + 8, clamped to the real plane
};
__device__ __forceinline__ ChromaRow10 load_chroma_row10(const uint8_t *row, int j0, int rw) {
  ChromaRow10 t;
  t.m = __ldg(reinterpret_cast<const uint2 *>(row + j0));
  t.l = __ldg(row + max(j0 - 1, 0));
  t.r = __ldg(row + min(j0 + 8, rw - 1));
  return t;
}
template <bool EDGE>
__device__ __forceinline__ void unpack_chroma_row10(const ChromaRow10 &t, int j0, int rw, int (&a)[10]) {
  a[0] = t.l;
#pragma unroll
  for (int k = 0; k < 8; k++) a[k + 1] = (int)(((k < 4 ? t.m.x : t.m.y) >> (8 * (k & 3))) & 0xffu);
  if (EDGE)
#pragma unroll
    for (int k = 1; k < 8; k++)  // past the real plane: its last sample, libjpeg's right edge
      if (j0 + k > rw - 1) a[k + 1] = a[k];
  a[9] = t.r;
}
// h2v1_fancy_upsample (V2 = false: `near` only) or h2v2_fancy_upsample of 8 chroma samples -> 16, packed into w[4].
template <bool V2, bool EDGE>
__device__ __forceinline__ void fancy16(const ChromaRow10 &nr, const ChromaRow10 &fr, int j0, int rw, uint32_t (&w)[4]) {
  int a[10];
  unpack_chroma_row10<EDGE>(nr, j0, rw, a);
  if (V2) {
    int f[10];
    unpack_chroma_row10<EDGE>(fr, j0, rw, f);
#pragma unroll
    for (int k = 0; k < 10; k++) a[k] = 3 * a[k] + f[k];  // column sums
  }
#pragma unroll
  for (int k = 0; k < 8; k++) {
    const int c3 = 3 * a[k + 1];
    const uint32_t lo = V2 ? (uint32_t)(c3 + a[k] + 8) >> 4 : (uint32_t)(c3 + a[k] + 1) >> 2;
    const uint32_t hi = V2 ? (uint32_t)(c3 + a[k + 2] + 7) >> 4 : (uint32_t)(c3 + a[k + 2] + 2) >> 2;
    if (k & 1) w[k >> 1] |= (lo | hi << 8) << 16;
    else w[k >> 1] = lo | hi << 8;
  }
}

template <bool PLANAR>  // PLANAR: planar 4:4:4 Y, U, V (HCJ_OUT_YUV444) instead of RGB24
__global__ void __launch_bounds__(128) k_rgb_libjpeg(DecodeBatchDev b) {
  const HcjImageDesc &d = b.descs[blockIdx.z + b.img_lo];
  if (!d.valid || !d.libjpeg) return;
  const int x0 = (blockIdx.x * blockDim.x + threadIdx.x) * 16, y = blockIdx.y;
  if (y >= d.height || x0 >= d.width) return;
  const int n = min(16, d.width - x0);
  const HcjCompGeom &gy = d.comp[0], &gu = d.comp[1], &gv = d.comp[2];
  const uint8_t *py = b.planes + gy.plane_off, *pu = b.planes + gu.plane_off, *pv = b.planes + gv.plane_off;
  const int hr = gu.up_h, vr = gu.up_v;
  const int rw = (d.width + hr - 1) / hr, rh = (d.height + vr - 1) / vr;  // the real chroma plane
  uint32_t wy[4], wu[4], wv[4];
  if (gy.up_h == 1 && gy.up_v == 1 && hr == 2 && vr <= 2 && gv.up_h == 2 && gv.up_v == vr && rw > 2) {
    const int j0 = x0 >> 1, i = y / vr;
    const int fi = vr == 2 ? min(max(i + ((y & 1) ? 1 : -1), 0), rh - 1) : i;
    load16(py + (size_t)y * gy.decoded_w + x0, wy);
    const ChromaRow10 un = load_chroma_row10(pu + (size_t)i * gu.decoded_w, j0, rw), vn = load_chroma_row10(pv + (size_t)i * gv.decoded_w, j0, rw);
    const ChromaRow10 uf = load_chroma_row10(pu + (size_t)fi * gu.decoded_w, j0, rw), vf = load_chroma_row10(pv + (size_t)fi * gv.decoded_w, j0, rw);
    const bool edge = j0 + 8 > rw - 1;
    if (vr == 2) {
      if (edge) fancy16<true, true>(un, uf, j0, rw, wu), fancy16<true, true>(vn, vf, j0, rw, wv);
      else fancy16<true, false>(un, uf, j0, rw, wu), fancy16<true, false>(vn, vf, j0, rw, wv);
    } else {
      if (edge) fancy16<false, true>(un, uf, j0, rw, wu), fancy16<false, true>(vn, vf, j0, rw, wv);
      else fancy16<false, false>(un, uf, j0, rw, wu), fancy16<false, false>(vn, vf, j0, rw, wv);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 4; k++) wy[k] = wu[k] = wv[k] = 0u;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      if (i >= n) break;
      const int x = x0 + i, sh = 8 * (i & 3);
      const HcjCompGeom *g[3] = {&gy, &gu, &gv};
      const uint8_t *p[3] = {py, pu, pv};
      uint32_t v[3];
#pragma unroll
      for (int c = 0; c < 3; c++) {
        const int h = g[c]->up_h, vv = g[c]->up_v;
        v[c] = (uint32_t)libjpeg_upsample(p[c], g[c]->decoded_w, (d.width + h - 1) / h, (d.height + vv - 1) / vv, h, vv, x, y);
      }
      wy[i >> 2] |= v[0] << sh;
      wu[i >> 2] |= v[1] << sh;
      wv[i >> 2] |= v[2] << sh;
    }
  }
  if (PLANAR) {
    const size_t plane = (size_t)d.width * d.height;
    uint8_t *oy = b.out + d.out_off + (size_t)y * d.width + x0;
    store_any<4>(oy, wy, n);
    store_any<4>(oy + plane, wu, n);
    store_any<4>(oy + 2 * plane, wv, n);
    return;
  }
  uint32_t o[12];
#pragma unroll
  for (int k = 0; k < 4; k++) {  // 4 pixels -> 12 bytes = 3 words
    uint32_t px[4];
#pragma unroll
    for (int i = 0; i < 4; i++)
      px[i] = ycc_to_rgb((wy[k] >> (8 * i)) & 0xff, (wu[k] >> (8 * i)) & 0xff, (wv[k] >> (8 * i)) & 0xff);
    o[3 * k + 0] = px[0] | (px[1] << 24);
    o[3 * k + 1] = (px[1] >> 8) | (px[2] << 16);
    o[3 * k + 2] = (px[2] >> 16) | (px[3] << 8);
  }
  store_any<12>(b.out + d.out_off + ((size_t)y * d.width + x0) * 3, o, 3 * n);
}

void launch_rgb(const DecodeBatchDev &b, bool planar444, cudaStream_t s) {
  if (b.img_hi <= b.img_lo || b.max_rgb_rows == 0) return;
  if (!planar444 && b.has_fused && b.max_blocks)
    k_rgb444_fix<<<dim3((b.max_blocks + 32 * 128 - 1) / (32 * 128), b.img_hi - b.img_lo), 128, 0, s>>>(b);
  if (!planar444 && b.has_fused_sub) {
    k_rgb_deferred<<<dim3((b.max_deferred_groups + 127) / 128, b.img_hi - b.img_lo), 128, 0, s>>>(b);
  }
  dim3 block(128);
  dim3 grid((b.max_width / 16 + 127 + 1) / 128, b.max_rgb_rows, b.img_hi - b.img_lo);
  if (b.has_444) {
    if (planar444) k_rgb<true, false><<<grid, block, 0, s>>>(b);
    else k_rgb<false, false><<<grid, block, 0, s>>>(b);
  }
  if (b.has_subsampled) {
    if (planar444) k_rgb<true, true><<<grid, block, 0, s>>>(b);
    else {
      if (b.has_subsampled & 1) k_rgb_sub_pairs<<<dim3(grid.x, (b.max_rgb_rows + 1) / 2, grid.z), block, 0, s>>>(b);
      if (b.has_subsampled & 2) k_rgb<false, true><<<grid, block, 0, s>>>(b);
    }
  }
  if (b.has_libjpeg) {
    if (planar444) k_rgb_libjpeg<true><<<grid, block, 0, s>>>(b);
    else k_rgb_libjpeg<false><<<grid, block, 0, s>>>(b);
  }
}

// `oyuv convert` (tools/src/oconv.ml:111-133): planar frame -> 4:4:4 (Planar_444.convert_from_420 / _422) -> Yuv.crop with
// edge clamp (yuv.ml:43-62) -> Planar_444.convert_to_420 / _422 (planar_444.ml:18-23,36-50,68-80,105-120), one
// output sample per thread, nothing materialised in between.
struct ConvertArgs {
  const uint8_t *src;
  uint8_t *dst;
  int sw, sh, schroma;  // source frame
  int dw, dh, dchroma;  // destination frame
  int x_off, y_off;     // position of the destination's origin in the source (crop)
};
__device__ __forceinline__ int conv_sample_444(const ConvertArgs &a, int c, int x, int y) {
  // sample (x, y) of plane c of the destination-sized 4:4:4 frame = the source's 4:4:4 frame at the clamped position
  x = min(max(x + a.x_off, 0), a.sw - 1);
  y = min(max(y + a.y_off, 0), a.sh - 1);
  if (c == 0) return a.src[(size_t)y * a.sw + x];
  const int hs_log = a.schroma == 444 ? 0 : 1, vs_log = a.schroma == 420 ? 1 : 0;
  const int cw = a.sw >> hs_log, ch = a.sh >> vs_log;
  const uint8_t *p = a.src + (size_t)a.sw * a.sh + (size_t)(c - 1) * cw * ch;
  return up_sample(p, cw, cw, ch, x, y, hs_log, vs_log);
}
__global__ void __launch_bounds__(256) k_yuv_convert(ConvertArgs a) {
  const int hs_log = a.dchroma == 444 ? 0 : 1, vs_log = a.dchroma == 420 ? 1 : 0;
  const int cw = a.dw >> hs_log, ch = a.dh >> vs_log;
  const size_t ny = (size_t)a.dw * a.dh, nc = (size_t)cw * ch;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ny + 2 * nc) return;
  int v;
  if (i < ny) {
    v = conv_sample_444(a, 0, (int)(i % a.dw), (int)(i / a.dw));
  } else {
    const int c = i < ny + nc ? 1 : 2;
    const size_t k = i - ny - (c - 1) * nc;
    const int x = (int)(k % cw), y = (int)(k / cw);
    if (hs_log && vs_log)
      v = (conv_sample_444(a, c, 2 * x, 2 * y) + conv_sample_444(a, c, 2 * x + 1, 2 * y) + conv_sample_444(a, c, 2 * x, 2 * y + 1) +
           conv_sample_444(a, c, 2 * x + 1, 2 * y + 1) + 2) >> 2;
    else if (hs_log)
      v = (conv_sample_444(a, c, 2 * x, y) + conv_sample_444(a, c, 2 * x + 1, y) + 1) >> 1;
    else
      v = conv_sample_444(a, c, x, y);
  }
  a.dst[i] = (uint8_t)v;
}
void launch_yuv_convert(const uint8_t *src, int sw, int sh, int schroma, int x_off, int y_off, uint8_t *dst, int dw, int dh, int dchroma,
                        cudaStream_t s) {
  ConvertArgs a{src, dst, sw, sh, schroma, dw, dh, dchroma, x_off, y_off};
  const size_t n = yuv_frame_bytes(dw, dh, dchroma);
  if (n) k_yuv_convert<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(a);
}
size_t yuv_frame_bytes(int w, int h, int chroma) {  // Frame.create (frame.ml:32-40)
  const size_t cw = chroma == 444 ? w : w / 2, ch = chroma == 420 ? h / 2 : h;
  return (size_t)w * h + 2 * cw * ch;
}

// Debug tap: Decoder.Component.Summary (decoder.ml:189-203) of `count` blocks of one image, from its coefficient
// blocks: position, predictor, coefs with the DC differential restored, dequant, idct (before clipping), recon.
// One thread per block, the model's 64-bit arithmetic verbatim.
__global__ void k_block_log(DecodeBatchDev b, uint32_t img, uint32_t first, uint32_t count, BlockLog *out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count) return;
  const HcjImageDesc &d = b.descs[img];
  const uint32_t blk = first + t, mcu = blk / d.bpm, j = blk - mcu * d.bpm;
  const int c = d.blk_comp[j];
  const HcjCompGeom &g = d.comp[c];
  const int16_t *cf = b.coefs + (d.coef_off + blk) * 64;
  int32_t pred = 0;  // the component's dc_pred before this block (decoder.ml:151-165; reset per restart interval)
  if (d.blk_bx[j] != 0 || d.blk_by[j] != 0) pred = cf[-64];
  else if (mcu != 0 && !(d.ri && mcu % d.ri == 0)) pred = b.coefs[(d.coef_off + (uint64_t)(mcu - 1) * d.bpm + g.first_blk + g.hs * g.vs - 1) * 64];
  BlockLog &o = out[t];
  o.x = (int32_t)((mcu % d.mcus_wide) * g.hs + d.blk_bx[j]) * 8;  // decoder.ml:353-360
  o.y = (int32_t)((mcu / d.mcus_wide) * g.vs + d.blk_by[j]) * 8;
  o.dc_pred = cf[0];
  o.component = c;
  const int32_t *q = b.qtables + d.qt_off + c * 128;
  int64_t w[64];
  for (int i = 0; i < 64; i++) {
    o.coefs[i] = i ? cf[i] : (int16_t)(cf[0] - pred);
    const int64_t v = (int64_t)cf[i] * q[i];  // decoder.ml:142-149 (the DC is dc_pred + coefs.(0) = the resolved value)
    w[zigzag_inverse(i)] = v;
  }
  for (int i = 0; i < 64; i++) o.dequant[i] = (int32_t)w[i];
  idct_8x8<int64_t>(w);
  for (int i = 0; i < 64; i++) {
    o.idct[i] = (int32_t)w[i];
    const int64_t sv = w[i] < -128 ? -128 : w[i] > 127 ? 127 : w[i];  // decoder.ml:213-224
    o.recon[i] = (uint8_t)(sv + 128);
  }
}
void launch_block_log(const DecodeBatchDev &b, uint32_t img, uint32_t first, uint32_t count, BlockLog *out, cudaStream_t s) {
  if (count) k_block_log<<<(count + 63) / 64, 64, 0, s>>>(b, img, first, count, out);
}

// Ocompare.square_error / max_difference (tools/src/ocompare.ml:8-52).
// res[0] = square error, res[1] = max difference, res[2] = total difference (Ocompare, tools/src/ocompare.ml:8-52)
__global__ void k_compare(const uint8_t *a, const uint8_t *bb, size_t n, unsigned long long *res) {
  unsigned long long acc = 0, tot = 0;
  int mx = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    int dlt = abs((int)a[i] - (int)bb[i]);
    acc += (unsigned long long)(dlt * dlt);
    tot += (unsigned long long)dlt;
    mx = max(mx, dlt);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, s);
    tot += __shfl_xor_sync(0xffffffffu, tot, s);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(res, acc);
    atomicMax(reinterpret_cast<int *>(res + 1), mx);
    atomicAdd(res + 2, tot);
  }
}

// The same per (image, plane) of a decoded batch against reference frames (hcj_batch_compare): grid (chunks, 4, images).
__global__ void __launch_bounds__(256) k_compare_planes(const uint8_t *out, const uint8_t *ref, const ComparePlane *planes,
                                                         unsigned long long *acc /* [images][4][4] */) {
  const ComparePlane pl = planes[blockIdx.z * 4 + blockIdx.y];
  if (pl.bytes == 0) return;
  const uint8_t *a = out + pl.out_off, *r = ref + pl.ref_off;
  unsigned long long se = 0, td = 0;
  unsigned mx = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < pl.bytes; i += (uint64_t)gridDim.x * blockDim.x) {
    const unsigned dlt = (unsigned)abs((int)a[i] - (int)r[i]);
    se += dlt * dlt;
    td += dlt;
    mx = max(mx, dlt);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, s);
    td += __shfl_xor_sync(0xffffffffu, td, s);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  }
  if ((threadIdx.x & 31) == 0) {
    unsigned long long *o = acc + ((size_t)blockIdx.z * 4 + blockIdx.y) * 4;
    atomicAdd(o + 0, se);
    atomicAdd(o + 1, td);
    atomicMax(o + 2, (unsigned long long)mx);
  }
}
void launch_compare_planes(const uint8_t *out, const uint8_t *ref, const ComparePlane *planes, unsigned long long *acc, int images,
                           cudaStream_t s) {
  if (images <= 0) return;
  k_compare_planes<<<dim3(32, 4, images), 256, 0, s>>>(out, ref, planes, acc);
}

void launch_compare(const uint8_t *a, const uint8_t *b, size_t n, unsigned long long *res, cudaStream_t s) {
  if (n == 0) return;
  size_t want = (n + 255) / 256;
  unsigned blocks = (unsigned)(want < 148 * 8 ? want : 148 * 8);
  k_compare<<<blocks, 256, 0, s>>>(a, b, n, res);
}

// Per-device launch configuration, done once per context right after cudaSetDevice (hcj_ctx_create): the opt-in to
// more than 48 KiB of dynamic shared memory is a per-device attribute of each kernel, so a process that drives
// several GPUs has to set it on every one of them (worst case over table sets: HCJ_MAX_COMP table pairs).
int configure_device(int *sm_count) {
  int dev = 0, sms = 148;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  DecodeBatchDev worst;
  worst.max_pairs = HCJ_MAX_COMP;
  const size_t base = ((sizeof(SmemTables) + 15) & ~size_t(15)) + ((sizeof(ScanCtx) + 15) & ~size_t(15)) + lut_smem_bytes(worst);
  const size_t stage = (HR_THREADS / 32) * HR_STAGE_WORDS * sizeof(uint32_t);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_huff_restart, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(base + stage));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_spec_sync, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(base + multi_smem_bytes(worst)));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_spec_fix, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)base);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(k_spec_write, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)(base + (SPEC_WRITE_THREADS / 32) * HR_STAGE_WORDS * sizeof(uint32_t)));
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<false, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(k_idct_persistent<false, 8, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IDCT_SMEM);
  if (sm_count) *sm_count = sms;
  return (int)e;
}

}  // namespace hcjk
