// hcj_kernels.cuh — launch wrappers of the CUDA kernels (hcj_kernels.cu), called by hcj_api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "hcj_common.h"

namespace hcjk {

struct DsTile;
struct IdctTile;

// Everything the decode kernels need about one batch resident in HBM.
struct DecodeBatchDev {
  int n;                          // images
  int sm_count;                   // SMs of the context's device (persistent grids)
  const HcjImageDesc *descs;      // [n]
  HcjImageState *states;          // [n]
  const uint8_t *files;           // compressed files, each starting at a 16-byte boundary
  uint8_t *entropy;               // destuffed entropy-coded bytes per image
  uint32_t *seg_offs;             // per image: nseg_expected + 1 byte offsets into its entropy bytes
  uint32_t *seg_sub;              // same indexing, speculatively decoded images with restart intervals: first subsequence of every interval (k_spec_units)
  struct DsTile *ds_tiles;        // per 4 KiB tile of every scan: counts, then offsets (k_destuff_*)
  uint32_t max_ds_tiles;          // max tiles of any image
  uint32_t total_ds_tiles;        // records in ds_tiles (zeroed before every decode: the look-back reads their status)
  const HcjTableSet *table_sets;
  const uint16_t *lut_primary;    // primary LUT pool
  const uint16_t *lut_full;       // full LUT pool
  const int32_t *qtables;         // quant tables pool, zig-zag order, one int32 per entry
  int16_t *coefs;                 // [total blocks][64], zig-zag, DC resolved
  // TMA tensor map of `coefs` as a 2-D uint16 tensor [total blocks][64], box = one IDCT tile (HCJ_IDCT_THREADS
  // blocks), 128-byte swizzle (a CUtensorMap: opaque 128 bytes, built by make_coef_tensor_map)
  alignas(64) unsigned char coef_map[128];
  uint32_t *wide_flags;           // 1 bit per block: take the 64-bit IDCT (zeroed before every decode)
  uint8_t *planes;                // padded planes (scratch for RGB mode, the output for PLANES mode)
  uint8_t *out;                   // outputs
  // launch geometry, computed on the host
  const uint32_t *list_restart;   // images decoded per restart interval
  int n_restart;
  uint32_t max_segments;          // max nseg_expected over list_restart
  uint32_t max_pairs;             // max (dc, ac) table pairs any image uses (sizes the LUT shared memory)
  const uint32_t *list_spec;      // images decoded speculatively (no restart markers)
  int n_spec;
  // per subsequence of those images (index = HcjImageDesc::sub_off + subsequence):
  uint16_t *sub_start;            // packed decoder state the subsequence was last decoded from
  uint16_t *sub_end2;             // packed state at its end (decoded from sub_start)
  uint32_t *sub_first;            // where the first MCU begun inside the subsequence starts, and the blocks begun in front of it
  int4 *sub_dpre;                 // DC differential sums of those blocks in front
  int32_t *sub_nstart;            // blocks begun
  int32_t *sub_blk;               // index (within the image) of the first of them: segmented exclusive prefix (k_spec_fix)
  int4 *sub_dc;                   // DC differential sums per scan component; after the scan: exclusive prefix
  uint32_t *sub_list;             // scratch: subsequences to decode again in the current fix-point round
  uint32_t max_sub_chunks;        // max over list_spec of ceil(subsequences / 256)
  uint32_t spec_guess_bits;       // bits in front of a subsequence that k_spec_sync decodes from a guessed state
  int spec_has_units;             // list_spec holds images with (long) restart intervals: k_spec_units runs
  uint32_t max_idct_tiles;        // max over images of tiles_per_row * mcus_high
  struct IdctTile *idct_plan;     // one record per IDCT tile of the batch (k_idct_plan), image after image
  uint32_t total_idct_tiles;
  uint32_t tile_lo, tile_hi;      // tiles of the images [img_lo, img_hi)
  int tile_mcus;                  // MCUs per IDCT tile (upper bound; per-image value derived in-kernel)
  int block_k;                    // samples per block side in the output planes: 8, or 8 / s for a scaled decode (HCJ_FLAG_SCALE_*)
  uint32_t max_rgb_rows;          // max image height (RGB mode)
  int has_444, has_subsampled;    // the batch holds 4:4:4 / sub-sampled images that go through k_rgb: which instances to launch
                                  // (has_subsampled: bit 0 = of even size, bit 1 = of odd size)
  int has_fused;                  // ... 4:4:4 images whose RGB24 is produced inside k_idct_persistent (HcjImageDesc::fused_rgb == 1)
  int has_fused_sub;              // ... sub-sampled images of even size likewise (fused_rgb == 2; k_rgb_deferred finishes them)
  uint32_t max_blocks;            // max blocks of any image
  uint32_t max_deferred_groups;   // max over fused sub-sampled images of the 16-pixel groups k_rgb_deferred converts
  uint32_t max_width;
  uint64_t total_blocks;
  // sub-range of the batch handled by one launch (the pipelined host path decodes chunk by chunk)
  uint32_t img_lo, img_hi;        // images [img_lo, img_hi)
  uint32_t lr_lo, lr_hi;          // entries of list_restart
  uint32_t ls_lo, ls_hi;          // entries of list_spec
  // HCJ_FLAG_LIBJPEG (kept behind the fields above so that their offsets, and the other kernels' code, stay as they were)
  int islow;                      // k_idct_persistent reconstructs with libjpeg's islow IDCT
  int has_libjpeg;                // the batch holds images that k_rgb_libjpeg up-samples (HcjImageDesc::libjpeg)
};

// Once per context, with its device current: shared-memory opt-ins of the kernels (a per-device attribute) and the
// SM count.  Returns a cudaError_t-compatible code.
int configure_device(int *sm_count);
// Clears what a decode pass expects to find cleared (wide-block flags, image states, destuff tile records); once per
// decode of the batch, before the first launch_destuff.  Returns a cudaError_t-compatible code.
int decode_prologue(const DecodeBatchDev &b, cudaStream_t s);
void launch_destuff(const DecodeBatchDev &b, cudaStream_t s);
int destuff_kernel_count();
void launch_huff_restart(const DecodeBatchDev &b, cudaStream_t s);
void launch_huff_spec(const DecodeBatchDev &b, cudaStream_t s);
int huff_spec_kernel_count(const DecodeBatchDev &b);
void launch_idct(const DecodeBatchDev &b, int mode, cudaStream_t s);
int idct_kernel_count();
size_t idct_plan_bytes(uint32_t tiles);
// Fills b->coef_map for b->coefs / b->total_blocks.  Returns a cudaError_t-compatible code (0 = ok).
int make_coef_tensor_map(DecodeBatchDev *b);
void launch_rgb(const DecodeBatchDev &b, bool planar444, cudaStream_t s);
void launch_idct_blocks(const int16_t *coefs, size_t nblocks, const uint16_t *qt, bool force_wide, uint8_t *out,
                        cudaStream_t s);
void launch_compare(const uint8_t *a, const uint8_t *b, size_t n, unsigned long long *res /* sse, max, total */, cudaStream_t s);

size_t yuv_frame_bytes(int w, int h, int chroma);
void launch_yuv_convert(const uint8_t *src, int sw, int sh, int schroma, int x_off, int y_off, uint8_t *dst, int dw, int dh, int dchroma,
                        cudaStream_t s);

struct BlockLog {  // = hcj_block_log (include/hcjpeg.h)
  int32_t x, y, dc_pred, component;
  int16_t coefs[64];
  int32_t dequant[64];
  int32_t idct[64];
  uint8_t recon[64];
};
void launch_block_log(const DecodeBatchDev &b, uint32_t img, uint32_t first, uint32_t count, BlockLog *out, cudaStream_t s);

struct ComparePlane {
  uint64_t out_off;  // plane in the batch output buffer
  uint64_t ref_off;  // the same plane in the uploaded reference frames
  uint64_t bytes;    // 0: no such plane
};
void launch_compare_planes(const uint8_t *out, const uint8_t *ref, const ComparePlane *planes, unsigned long long *acc, int images,
                           cudaStream_t s);

// ---- encoder ----
constexpr int HCJ_ENC_SLOT_WORDS = 16;  // blocks of up to 512 bits are packed once (k_block_bits) and only shifted into place (k_place)
struct EncodeBatchDev {
  int n;                      // frames
  int ncomp, bpm;
  int hs[3], vs[3];
  int plane_w[3], plane_h[3]; // padded geometry (never materialised: reads outside src are 0)
  int src_w[3], src_h[3];
  uint64_t src_off[3];        // offset of each source plane inside one frame
  uint64_t frame_bytes;       // bytes of one source frame
  int mcus_wide, mcus_high;
  int linear_blit;            // monochrome: the source plane is copied linearly into the padded plane (encode_monochrome)
  uint32_t nblocks;           // per frame
  uint32_t restart_interval;  // 0 = none
  uint32_t nseg;              // segments per frame (1 if no restart)
  uint32_t seg_chunks;        // byte-stuffing work units per segment (a lone segment is cut into 1 KiB chunks)
  uint8_t blk_comp[HCJ_MAX_BPM + 2], blk_bx[HCJ_MAX_BPM + 2], blk_by[HCJ_MAX_BPM + 2];
  const uint8_t *src;         // [n] frames
  const uint16_t *qt;         // [2][64] zig-zag
  const uint32_t *qrecip;     // [2][64] reciprocals of 4q
  const uint32_t *dc_codes;   // [2][16]  (bits << 8) | length
  const uint32_t *ac_codes;   // [2][256]
  int16_t *quant;             // [n][nblocks][64] zig-zag, DC absolute
  uint32_t *blk_bits;         // [n][nblocks] bit length of each block's code, later exclusive offsets per segment
  uint32_t *blk_words;        // [n][nblocks][HCJ_ENC_SLOT_WORDS] every block's own bit string, first bit in bit 31 of word 0 (k_block_bits)
  uint32_t *seg_bytes;        // [n][nseg * seg_chunks + 1] stuffed byte length of every unit, later exclusive offsets
  uint8_t *raw;               // [n][raw_stride] unstuffed packed bits, segments byte-aligned
  uint64_t raw_stride;
  uint8_t *out;               // [n][out_stride] finished files
  uint64_t out_stride;
  uint32_t *out_len;          // [n]
  uint32_t *long_blocks;      // != 0: some block of the chunk is longer than its slot (k_pack has work)
  const uint8_t *header;      // shared header bytes
  uint32_t header_len;
};
void launch_encode(const EncodeBatchDev &e, cudaStream_t s);
void launch_encode_block_log(const EncodeBatchDev &e, uint32_t first, uint32_t count, void *out /* hcj_encoder_block[count] */, cudaStream_t s);
int encode_kernel_count();
// K10: RGB24 frames (device pointer table rgb[frames]) -> planar frames of `chroma` (420 / 422 / 444 / 400), back to back in dst
void launch_rgb_to_ycc(const uint8_t *const *rgb, int frames, int w, int h, int chroma, uint8_t *dst, cudaStream_t s);
uint64_t rgb_frame_planar_bytes(int w, int h, int chroma);

}  // namespace hcjk
