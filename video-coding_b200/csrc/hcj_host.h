// hcj_host.h — host-side (CPU, C++) half of the drop-in: header parsing, geometry and table
// construction.  These are the cheap, sequential, data-dependent steps the model performs before its
// per-block loop (Decoder.Header.decode, Decoder.init); everything from extract_entropy_coded_bits
// down runs on the device.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/hcjpeg.h"
#include "hcj_common.h"

namespace hcj {

// Decoder.Header.decode (decoder.ml:37-70) over a From_string bit reader.
// clear_tables = false leaves the unused quant / Huffman table slots of `out` as they were (batch path).
int header_decode(const uint8_t *jpeg, size_t len, hcj_header *out, unsigned flags = 0, bool clear_tables = true);

// Frame boundaries of a Motion-JPEG stream (whole files back to back).
int mjpeg_split(const uint8_t *stream, size_t len, size_t *offsets, size_t *lengths, int capacity, int *nframes);

// Decoder.init geometry (decoder.ml:304-345) + which tables each scan component binds to.
struct ImagePlan {
  hcj_frame_info info;
  int qt_index[HCJ_MAX_COMPONENTS];       // index into header.quant_tables (list order)
  int dc_index[HCJ_MAX_COMPONENTS];       // index into header.huffman_tables
  int ac_index[HCJ_MAX_COMPONENTS];
  int blk_comp[HCJ_MAX_BPM], blk_bx[HCJ_MAX_BPM], blk_by[HCJ_MAX_BPM];
  // libjpeg's up-sampling ratios (h_max / h_c, v_max / v_c), all components integral; HCJ_FLAG_LIBJPEG only
  bool up_integral;
  int up_h[HCJ_MAX_COMPONENTS], up_v[HCJ_MAX_COMPONENTS];
};
int plan_image(const hcj_header &h, unsigned flags, ImagePlan *plan);
// HCJ_FLAG_SCALE_*: log2 of the scale denominator s (0 = full size, 1..3 = 1/2, 1/4, 1/8)
inline int scale_log2(unsigned flags) { return (int)((flags & HCJ_FLAG_SCALE_MASK) >> 4); }

// Tables.Specification.create_code_table + Tables.Lut.create (tables.ml:27-51,478-502), re-packed as
// a HCJ_LUT_BITS primary table plus the model's full 2^max_bits table.
struct HuffLut {
  int max_bits = 0;
  std::vector<uint16_t> full;     // 2^max_bits entries: (length << 8) | data, 0 = None
  std::vector<uint16_t> primary;  // HCJ_LUT_ENTRIES entries: primary table, then HCJ_LUT_NSUB sub-tables
};
int build_lut(const hcj_dht &t, HuffLut *lut);

// Defaults of the encoder (Tables.Default, tables.ml:54-476; Quant_tables, quant_tables.ml).
void default_spec(int which /*0 dc_luma 1 dc_chroma 2 ac_luma 3 ac_chroma*/, const uint8_t **lengths,
                  const uint8_t **values, int *nvalues);
void quant_scale(bool chroma, int quality, uint16_t out[64]);

// Tables.Encoder.dc_table / ac_table (tables.ml:504-545) flattened for the device:
// code[(run << 4) | size] = (bits << 8) | length  (length 0 = no such code); dc uses run = 0.
void encoder_tables(int which_dc, int which_ac, uint32_t dc[16], uint32_t ac[256]);

// Encoder.Parameters (encoder.ml:287-369) for 420 / 422 / 444.
struct EncodePlan {
  int width, height, chroma, quality, restart_interval;
  int ncomp, bpm;
  int hs[3], vs[3];
  int plane_w[3], plane_h[3];   // padded planes, encoder.ml:450-463
  int src_w[3], src_h[3];       // Frame.create plane sizes, frame.ml:32-40
  int mcus_wide, mcus_high;
  int64_t nblocks;
  uint16_t qt[2][64];
  int blk_comp[HCJ_MAX_BPM], blk_bx[HCJ_MAX_BPM], blk_by[HCJ_MAX_BPM];
};
int plan_encode(int width, int height, int chroma, int quality, int restart_interval, EncodePlan *p);
// Encoder.write_headers (encoder.ml:371-418); appends to `out`.
void write_headers(const EncodePlan &p, std::vector<uint8_t> *out);

}  // namespace hcj
