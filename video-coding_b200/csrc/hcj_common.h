// hcj_common.h — structures shared by the host side (hcj_host.cpp, hcj_api.cu) and the kernels.
//
// Vocabulary follows the reference model: MCU ("macroblock" in decoder.ml:374-383), block (8x8),
// scan component, restart interval ("segment" here: an independently decodable run of MCUs whose
// entropy-coded bits start byte-aligned with all DC predictors at 0).
#pragma once
#include <stdint.h>

#define HCJ_LUT_BITS 10                    // primary Huffman LUT index width
#define HCJ_LUT_SIZE (1 << HCJ_LUT_BITS)
#define HCJ_LUT_NSUB 8                     // second-level sub-tables per Huffman table (shared memory)
#define HCJ_LUT_SUB_BITS 6                 // each covers the 16 - HCJ_LUT_BITS bits below an unresolved prefix
#define HCJ_LUT_SUB_SIZE (1 << HCJ_LUT_SUB_BITS)
#define HCJ_LUT_ENTRIES (HCJ_LUT_SIZE + HCJ_LUT_NSUB * HCJ_LUT_SUB_SIZE)  // per table, uint16 each
#define HCJ_MAX_BPM 10                     // blocks per MCU (T.81 limit)
#define HCJ_MAX_COMP 4
#ifndef HCJ_IDCT_THREADS
#define HCJ_IDCT_THREADS 128              // threads (= blocks) per IDCT tile
#endif
#ifndef HCJ_IDCT_CTAS_PER_SM
#define HCJ_IDCT_CTAS_PER_SM 5                 // 96 registers: measured best (4 -> 3.09 ms, 5 -> 2.92 ms, 6 -> 3.99 ms with blocks in local memory)
#endif

// Internal status values produced on the device (same numbering as include/hcjpeg.h).
#define HCJ_DEV_OK 0
#define HCJ_DEV_NO_DC_CODE (-2)
#define HCJ_DEV_NO_AC_CODE (-3)
#define HCJ_DEV_COEF_INDEX (-4)
#define HCJ_DEV_BITS_OOB (-9)
#define HCJ_DEV_NO_TERMINATOR (-20)
#define HCJ_DEV_RESTART_COUNT (-21)
#define HCJ_DEV_DC_RANGE (-23)

// One Huffman table as the kernels see it.
//   primary[i] (i = next HCJ_LUT_BITS bits): (length << 8) | data;
//                0x8000 | k = "longer code: look in sub-table k"; 0 = "not resolved here"
//   sub-table k (HCJ_LUT_SUB_SIZE entries, indexed by the max_bits - HCJ_LUT_BITS bits that follow the
//                prefix): same encoding as the full table
//   full table (2^max_bits entries, (length << 8) | data, 0 = None in Tables.Lut, tables.ml:492) lives in
//   global memory at full_off and is consulted only when the primary entry is 0 (tables with more than
//   HCJ_LUT_NSUB unresolved prefixes; never the case for the Annex K tables).
struct HcjTableMeta {
  uint32_t full_off;  // offset (in uint16 entries) into the batch's full-LUT pool
  uint32_t max_bits;  // Tables.Lut.max_bits (tables.ml:491)
};

// A table set = the (dc, ac) pairs used by the scan components of one image, de-duplicated.
struct HcjTableSet {
  HcjTableMeta meta[HCJ_MAX_COMP][2];  // [pair][0 = dc, 1 = ac]
  uint32_t primary_off;                // offset (uint16 entries) of lut[pair][dc/ac][HCJ_LUT_ENTRIES]
  uint32_t npairs;
};

struct HcjCompGeom {
  int32_t hs, vs;                 // sampling factors
  int32_t decoded_w, decoded_h;   // padded plane (decoder.ml:312-317)
  int32_t actual_w, actual_h;     // cropped plane (decoder.ml:318-323)
  int32_t pair;                   // index into the table set
  int32_t qt;                     // index into the image's quant tables (qt_off + 64 * qt)
  int32_t first_blk;              // first block-in-MCU index of this component
  uint8_t up_h, up_v;             // HCJ_FLAG_LIBJPEG, RGB24 / YUV444: up-sampling ratios h_max / h_c, v_max / v_c
  uint16_t pad_;
  uint64_t plane_off;             // byte offset of the padded plane in the batch plane buffer
  uint64_t out_off;               // byte offset of this component's plane in the image's output
};

struct HcjImageDesc {
  // compressed input
  uint64_t file_off;     // byte offset in the batch file buffer (multiple of 16)
  uint32_t file_len;
  uint32_t scan_start;   // first entropy-coded byte within the file
  // destuffed entropy-coded segment(s)
  uint64_t ent_off;      // byte offset in the batch entropy buffer (multiple of 16)
  uint32_t ent_cap;      // capacity in bytes
  uint32_t seg_off;      // index into the batch segment-offset array (nseg_expected + 1 entries)
  uint32_t nseg_expected;// ceil(nmcu / ri), or 1
  uint32_t ri;           // restart interval in MCUs (0 = none / pure model semantics)
  // geometry
  int32_t ncomp, bpm;
  int32_t mcus_wide, mcus_high;
  uint32_t nmcu, nblocks;
  uint64_t coef_off;     // first block of this image in the batch coefficient buffer
  HcjCompGeom comp[HCJ_MAX_COMP];
  uint8_t blk_comp[HCJ_MAX_BPM + 2];  // block-in-MCU -> scan component
  uint8_t blk_bx[HCJ_MAX_BPM + 2];    // block-in-MCU -> x within the component's MCU footprint
  uint8_t blk_by[HCJ_MAX_BPM + 2];
  uint8_t wide_idct;     // 1: some quant entry > 255 -> always take the 64-bit IDCT
  uint8_t valid;         // 0: header/geometry failed on the host; kernels skip the image
  uint8_t fused_rgb;     // RGB24 output, no 16-bit quant entries: k_idct_persistent converts to RGB itself (1 = 4:4:4, 2 = 4:2:0 / 4:2:2 of even size)
  uint8_t libjpeg;       // HCJ_FLAG_LIBJPEG, RGB24 / YUV444, not 4:4:4: k_rgb_libjpeg up-samples it (comp[].up_h / up_v)
  uint32_t table_set;    // index into the batch table sets
  uint32_t qt_off;       // offset (uint16 entries) of this image's quant tables [nqt][64], zig-zag order
  // output
  uint64_t out_off;      // byte offset of this image in the batch output buffer
  uint64_t out_bytes;
  int32_t chroma;        // 420 / 422 / 444 / 0
  int32_t width, height;
  uint32_t sub_bits;     // scans without restart markers: subsequence length in bits (a multiple of 32)
  uint32_t sub_off;      // index of the image's first subsequence record in the batch arrays
  uint32_t ds_off;       // index of the image's first destuff tile record
  uint32_t idct_tile_off;// index of the image's first IDCT tile in the batch tile plan
  uint32_t idct_tiles;   // tiles of this image (tiles per MCU row x MCU rows; 0 for an invalid image)
};

// Written by the destuff kernel, read by the decode kernels and fetched for debugging.
struct HcjImageState {
  uint32_t ent_len;    // destuffed bytes (all segments)
  uint32_t nseg_found;
  int32_t status;      // error found while destuffing (0 = ok)
  uint32_t pad_;
  // Earliest entropy-decode error in stream order: (bit position << 8) | -status, ~0 = none.  The
  // model raises at the first bad symbol it meets; threads race, so the minimum key decides.
  unsigned long long err_key;
};
#define HCJ_NO_ERR_KEY 0xffffffffffffffffull
