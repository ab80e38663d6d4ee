// hcj_host.cpp — host half of the drop-in (see hcj_host.h).  Pure C++, no CUDA.
//
// Restates, independently of oracle/, the parts of the model that stay on the CPU:
//   Bitstream_reader.From_string   common/src/bitstream_reader.ml:6-57
//   Decoder.Header.decode          jpeg/model/src/decoder.ml:5-71
//   Markers.*.decode               jpeg/model/src/markers.ml
//   Decoder.init (geometry)        jpeg/model/src/decoder.ml:294-345
//   Tables.Specification / Lut     jpeg/model/src/tables.ml:27-51,478-502
//   Encoder.Parameters / headers   jpeg/model/src/encoder.ml:207-264,287-418
#include "hcj_host.h"

#include <stddef.h>
#include <string.h>

#include <algorithm>

namespace hcj {

namespace {

struct Raise {
  int code;
};

// MSB-first cursor; bytes past the end read as zero (bitstream_reader.ml:19-22); `show n` raises
// iff n >= total bits (:32).  n <= 16 everywhere on this path.
class Bits {
 public:
  Bits(const uint8_t *buf, size_t len) : buf_(buf), len_(len) {}
  uint32_t show(int n) const {
    if ((uint64_t)n >= (uint64_t)len_ * 8) throw Raise{HCJ_ERR_BITS_OUT_OF_BOUNDS};
    // the n <= 16 bits at pos_ lie inside the three bytes from pos_ / 8 on (bytes past the end read as zero):
    // the same value as the model's bit-by-bit loop
    const uint64_t byte_no = pos_ >> 3;
    uint32_t w = 0;
    for (int k = 0; k < 3; k++) w = (w << 8) | (byte_no + k < len_ ? buf_[byte_no + k] : 0u);
    return n ? (w >> (24 - (pos_ & 7) - n)) & ((1u << n) - 1u) : 0u;
  }
  uint32_t get(int n) {
    uint32_t v = show(n);
    pos_ += n;
    return v;
  }
  void advance(uint64_t n) { pos_ += n; }
  void align_to_byte() {
    if (pos_ & 7) pos_ += 8 - (pos_ & 7);
  }
  uint64_t bit_pos() const { return pos_; }
  uint64_t length_in_bits() const { return (uint64_t)len_ * 8; }

 private:
  uint32_t bit(uint64_t p) const {
    uint64_t byte_no = p >> 3;
    uint32_t b = byte_no < len_ ? buf_[byte_no] : 0;
    return (b >> (7 - (p & 7))) & 1;
  }
  const uint8_t *buf_;
  size_t len_;
  uint64_t pos_ = 0;
};

enum : int {
  SOF0 = 0xc0, DHT = 0xc4, RST0 = 0xd0, SOI = 0xd8, EOI = 0xd9, SOS = 0xda, DQT = 0xdb, DRI = 0xdd,
  APP0 = 0xe0, APP15 = 0xef, COM = 0xfe
};

void find_marker(Bits &b) {  // decoder.ml:24-29
  b.align_to_byte();
  for (;;) {
    if (b.bit_pos() >= b.length_in_bits()) throw Raise{HCJ_ERR_TRUNCATED};  // the model never returns here
    if (b.get(8) == 0xff) return;
  }
}

template <class T>
void push_front(T *arr, int *n, const T &v) {  // OCaml list cons: newest first
  if (*n == HCJ_MAX_TABLE_SEGMENTS) throw Raise{HCJ_ERR_UNSUPPORTED_GEOMETRY};
  for (int i = *n; i > 0; i--) arr[i] = arr[i - 1];
  arr[0] = v;
  (*n)++;
}

// flags & HCJ_FLAG_T81_TABLES (stated extension): DQT / DHT segments hold as many tables as their length covers and
// parsing continues at the end of the segment; 0xFF fill bytes in front of a marker code are skipped.
void decode_impl(Bits &b, hcj_header *h, unsigned flags, bool clear_tables) {  // decoder.ml:37-70
  const bool t81 = (flags & HCJ_FLAG_T81_TABLES) != 0;
  if (clear_tables) {
    memset(h, 0, sizeof(*h));
  } else {  // batch path: the 64 + 64 table slots (38 KB) are written when a table is pushed; only the rest is cleared
    memset(h, 0, offsetof(hcj_header, quant_tables));
    h->n_huffman_tables = 0;
    h->scan_byte_pos = 0;
  }
  for (;;) {
    find_marker(b);
    int code = (int)b.get(8);
    while (t81 && code == 0xff && b.bit_pos() < b.length_in_bits()) code = (int)b.get(8);
    if (code == SOF0) {  // markers.ml:49-59
      h->has_frame = 1;
      h->sof_length = b.get(16);
      h->sample_precision = b.get(8);
      h->height = b.get(16);
      h->width = b.get(16);
      h->number_of_components = b.get(8);
      if (h->number_of_components > HCJ_MAX_COMPONENTS) throw Raise{HCJ_ERR_UNSUPPORTED_GEOMETRY};
      for (int i = 0; i < h->number_of_components; i++) {  // markers.ml:15-25
        hcj_component &c = h->components[i];
        c.identifier = b.get(8);
        c.horizontal_sampling_factor = b.get(4);
        c.vertical_sampling_factor = b.get(4);
        c.quantization_table_identifier = b.get(8);
      }
    } else if (code == SOS) {  // markers.ml:111-129
      h->has_scan = 1;
      h->sos_length = b.get(16);
      h->number_of_image_components = b.get(8);
      if (h->number_of_image_components > HCJ_MAX_COMPONENTS) throw Raise{HCJ_ERR_UNSUPPORTED_GEOMETRY};
      for (int i = 0; i < h->number_of_image_components; i++) {  // markers.ml:84-89
        hcj_scan_component &s = h->scan_components[i];
        s.selector = b.get(8);
        s.dc_coef_selector = b.get(4);
        s.ac_coef_selector = b.get(4);
      }
      h->start_of_predictor_selection = b.get(8);
      h->end_of_predictor_selection = b.get(8);
      h->successive_approximation_bit_high = b.get(4);
      h->successive_approximation_bit_low = b.get(4);
      h->scan_byte_pos = (int64_t)(b.bit_pos() >> 3);
      return;
    } else if (code == DQT) {  // markers.ml:162-168 — one table per segment (more with HCJ_FLAG_T81_TABLES)
      const uint64_t seg_end = b.bit_pos() + 8ull * b.show(16);
      const int seg_len = (int)b.get(16);
      do {
        hcj_dqt q;
        memset(&q, 0, sizeof(q));
        q.length = seg_len;
        int pq = b.get(4);
        if (pq > 1) throw Raise{HCJ_ERR_UNSUPPORTED_GEOMETRY};
        q.element_precision = 8 << pq;
        q.table_identifier = b.get(4);
        for (int i = 0; i < 64; i++) q.elements[i] = (int)b.get(q.element_precision);
        push_front(h->quant_tables, &h->n_quant_tables, q);
      } while (t81 && b.bit_pos() < seg_end);
      if (t81 && b.bit_pos() < seg_end) b.advance(seg_end - b.bit_pos());
    } else if (code == DHT) {  // markers.ml:210-220 — one table per segment (more with HCJ_FLAG_T81_TABLES)
      const uint64_t seg_end = b.bit_pos() + 8ull * b.show(16);
      const int seg_len = (int)b.get(16);
      do {
        hcj_dht t;
        memset(&t, 0, sizeof(t));
        t.length = seg_len;
        t.table_class = b.get(4);
        t.destination_identifier = b.get(4);
        int total = 0;
        for (int i = 0; i < 16; i++) {
          t.lengths[i] = b.get(8);
          total += t.lengths[i];
        }
        if (total > 256) throw Raise{HCJ_ERR_BAD_HUFFMAN_TABLE};
        t.nvalues = total;
        for (int i = 0; i < total; i++) t.values[i] = (uint8_t)b.get(8);
        push_front(h->huffman_tables, &h->n_huffman_tables, t);
      } while (t81 && b.bit_pos() < seg_end);
      if (t81 && b.bit_pos() < seg_end) b.advance(seg_end - b.bit_pos());
    } else if (code == DRI) {  // markers.ml:193-197
      h->has_restart_interval = 1;
      h->dri_length = b.get(16);
      h->restart_interval = b.get(16);
    } else if (code == SOI) {
      // keep scanning
    } else if ((code >= APP0 && code <= APP15) || code == COM) {  // skip, decoder.ml:31-34
      uint32_t len = b.show(16);
      b.advance((uint64_t)len * 8);
    } else {
      throw Raise{HCJ_ERR_UNSUPPORTED_MARKER};
    }
  }
}

int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

}  // namespace

int header_decode(const uint8_t *jpeg, size_t len, hcj_header *out, unsigned flags, bool clear_tables) {
  Bits b(jpeg, len);
  try {
    decode_impl(b, out, flags, clear_tables);
  } catch (const Raise &r) {
    return r.code;
  }
  return HCJ_OK;
}

// Motion JPEG: frames are whole JPEG files back to back.  A frame starts at FF D8; its header segments are stepped
// over by their length fields up to SOS; the entropy-coded bytes run to the first marker that is neither a stuffed
// FF 00, a fill FF, nor RSTn; the frame ends behind the EOI that follows (further segments, e.g. more scans of a
// file the decoder would reject anyway, are stepped over the same way).  Bytes between frames are skipped, and so
// is a would-be frame whose length fields do not lead from marker to marker.
int mjpeg_split(const uint8_t *s, size_t len, size_t *offsets, size_t *lengths, int capacity, int *nframes) {
  int n = 0;
  size_t p = 0;
  while (p + 1 < len) {
    const uint8_t *q = (const uint8_t *)memchr(s + p, 0xff, len - 1 - p);
    if (!q) break;
    p = (size_t)(q - s);
    if (s[p + 1] != 0xd8) {
      p++;
      continue;
    }
    const size_t start = p;
    p += 2;
    bool done = false, ok = false;
    while (!done && p + 1 < len) {
      if (s[p] != 0xff) {  // a length field led somewhere else than to a marker: not a frame, look for the next SOI
        done = true;
        p = start + 2;
        break;
      }
      const int code = s[p + 1];
      if (code == 0xff) {  // fill byte
        p++;
      } else if (code == 0xd9) {  // EOI
        p += 2;
        done = ok = true;
      } else if (code == 0xd8) {  // a new SOI before EOI: the frame was cut short
        done = true;
      } else if (code == 0x00 || (code >= 0xd0 && code <= 0xd7) || code == 0x01) {  // stuffed byte / RSTn / TEM: no length
        p += 2;
      } else {
        if (p + 3 >= len) break;
        const size_t seg = ((size_t)s[p + 2] << 8) | s[p + 3];
        p += 2 + seg;
        if (code == 0xda) {  // SOS: entropy-coded data follows, up to the next real marker
          while (p + 1 < len) {
            const uint8_t *r = (const uint8_t *)memchr(s + p, 0xff, len - 1 - p);
            if (!r) {
              p = len;
              break;
            }
            p = (size_t)(r - s);
            const int c2 = s[p + 1];
            if (c2 == 0x00 || (c2 >= 0xd0 && c2 <= 0xd7)) p += 2;
            else if (c2 == 0xff) p++;
            else break;
          }
        }
      }
    }
    if (ok) {
      if (n < capacity && offsets && lengths) {
        offsets[n] = start;
        lengths[n] = p - start;
      }
      n++;
    } else if (!done) {
      break;  // ran off the end inside a frame
    }
  }
  *nframes = n;
  return n > capacity && offsets ? HCJ_ERR_BUFFER_TOO_SMALL : HCJ_OK;
}

int plan_image(const hcj_header &h, unsigned flags, ImagePlan *plan) {
  memset(plan, 0, sizeof(*plan));
  hcj_frame_info &f = plan->info;
  // HCJ_FLAG_LIBJPEG with a scaled decode: libjpeg reconstructs chroma at another block size there (not implemented)
  if ((flags & HCJ_FLAG_LIBJPEG) && (flags & HCJ_FLAG_SCALE_MASK)) return HCJ_ERR_INVALID_ARG;
  if (!h.has_frame || !h.has_scan) return HCJ_ERR_NO_FRAME_OR_SCAN;  // decoder.ml:283-292
  int max_h = 0, max_v = 0;                                          // decoder.ml:294-302
  for (int i = 0; i < h.number_of_components; i++) {
    max_h = std::max(max_h, h.components[i].horizontal_sampling_factor);
    max_v = std::max(max_v, h.components[i].vertical_sampling_factor);
  }
  int ncomp = h.number_of_image_components;
  if (ncomp < 1 || ncomp > HCJ_MAX_COMPONENTS || max_h < 1 || max_v < 1 || max_h > 4 || max_v > 4)
    return HCJ_ERR_UNSUPPORTED_GEOMETRY;
  int64_t rounded_w = round_up(h.width, (int64_t)max_h * 8);  // decoder.ml:307-308
  int64_t rounded_h = round_up(h.height, (int64_t)max_v * 8);
  f.width = h.width;
  f.height = h.height;
  f.ncomp = ncomp;
  int bpm = 0;
  for (int i = 0; i < ncomp; i++) {
    const hcj_component *c = nullptr;  // find_component, decoder.ml:226-230
    for (int j = 0; j < h.number_of_components; j++)
      if (h.components[j].identifier == h.scan_components[i].selector) {
        c = &h.components[j];
        break;
      }
    if (!c) return HCJ_ERR_NO_COMPONENT;
    if (c->horizontal_sampling_factor < 1 || c->vertical_sampling_factor < 1) return HCJ_ERR_UNSUPPORTED_GEOMETRY;
    f.hs[i] = c->horizontal_sampling_factor;
    f.vs[i] = c->vertical_sampling_factor;
    f.decoded_width[i] = (int)(rounded_w * f.hs[i] / max_h);  // decoder.ml:312-323
    f.decoded_height[i] = (int)(rounded_h * f.vs[i] / max_v);
    f.actual_width[i] = (int)((int64_t)h.width * f.hs[i] / max_h);
    f.actual_height[i] = (int)((int64_t)h.height * f.vs[i] / max_v);
    plan->qt_index[i] = -1;  // find_quant_table, decoder.ml:232-236 (List.find: newest wins)
    for (int j = 0; j < h.n_quant_tables; j++)
      if (h.quant_tables[j].table_identifier == c->quantization_table_identifier) {
        plan->qt_index[i] = j;
        break;
      }
    if (plan->qt_index[i] < 0) return HCJ_ERR_NO_QUANT_TABLE;
    plan->dc_index[i] = plan->ac_index[i] = -1;  // find_huffman_table, decoder.ml:238-245
    for (int j = 0; j < h.n_huffman_tables; j++) {
      const hcj_dht &t = h.huffman_tables[j];
      if (plan->dc_index[i] < 0 && t.table_class == 0 && t.destination_identifier == h.scan_components[i].dc_coef_selector)
        plan->dc_index[i] = j;
    }
    if (plan->dc_index[i] < 0) return HCJ_ERR_NO_HUFFMAN_TABLE;
    for (int j = 0; j < h.n_huffman_tables; j++) {
      const hcj_dht &t = h.huffman_tables[j];
      if (plan->ac_index[i] < 0 && t.table_class == 1 && t.destination_identifier == h.scan_components[i].ac_coef_selector)
        plan->ac_index[i] = j;
    }
    if (plan->ac_index[i] < 0) return HCJ_ERR_NO_HUFFMAN_TABLE;
    for (int y = 0; y < f.vs[i]; y++)  // decode_component_seq order, decoder.ml:362-372
      for (int x = 0; x < f.hs[i]; x++) {
        if (bpm >= HCJ_MAX_BPM) return HCJ_ERR_UNSUPPORTED_GEOMETRY;
        plan->blk_comp[bpm] = i;
        plan->blk_bx[bpm] = x;
        plan->blk_by[bpm] = y;
        bpm++;
      }
  }
  f.blocks_per_mcu = bpm;
  f.mcus_wide = f.decoded_width[0] / (8 * f.hs[0]);  // decoder.ml:377-383
  f.mcus_high = f.decoded_height[0] / (8 * f.vs[0]);
  f.nblocks = (int64_t)f.mcus_wide * f.mcus_high * bpm;
  // The model writes block (x, y) of every component through a bounds-checked Plane (plane.ml:55-61).
  // Components whose sampling factors do not divide the maxima can fall outside their plane.
  for (int i = 0; i < ncomp; i++)
    if (f.mcus_wide * f.hs[i] * 8 > f.decoded_width[i] || f.mcus_high * f.vs[i] * 8 > f.decoded_height[i])
      return HCJ_ERR_PLANE_BOUNDS;
  f.restart_interval = ((flags & HCJ_FLAG_RESTART_EXT) && h.has_restart_interval) ? h.restart_interval : 0;
  // Scaled decode (HCJ_FLAG_SCALE_*): the frame of ceil(w / s) x ceil(h / s) with the same sampling factors, padded
  // planes of decoded_* / s (multiples of 8 / s: they hold every block's k x k samples); the block geometry above stays.
  const int scale_log = hcj::scale_log2(flags);
  if (scale_log) {
    const int s = 1 << scale_log;
    f.width = (h.width + s - 1) >> scale_log;
    f.height = (h.height + s - 1) >> scale_log;
    for (int i = 0; i < ncomp; i++) {
      f.decoded_width[i] >>= scale_log;
      f.decoded_height[i] >>= scale_log;
      f.actual_width[i] = (int)((int64_t)f.width * f.hs[i] / max_h);
      f.actual_height[i] = (int)((int64_t)f.height * f.vs[i] / max_v);
    }
  }
  f.planes_bytes = 0;
  for (int i = 0; i < ncomp; i++) f.planes_bytes += (size_t)f.decoded_width[i] * f.decoded_height[i];
  // get_yuv_frame -> Frame.of_planes -> infer_chroma_subsampling (frame.ml:42-61)
  f.chroma = 0;
  if (ncomp >= 3) {
    int yw = f.actual_width[0], yh = f.actual_height[0], uw = f.actual_width[1], uh = f.actual_height[1];
    if (uw == f.actual_width[2] && uh == f.actual_height[2]) {
      if (yw / 2 == uw && yh / 2 == uh) f.chroma = 420;
      else if (yw / 2 == uw && yh == uh) f.chroma = 422;
      else if (yw == uw && yh == uh) f.chroma = 444;
    }
  }
  if (f.chroma) {
    f.yuv_bytes = 0;
    for (int i = 0; i < 3; i++) f.yuv_bytes += (size_t)f.actual_width[i] * f.actual_height[i];
    f.rgb_bytes = (size_t)f.width * f.height * 3;
  }
  // HCJ_FLAG_LIBJPEG: jdsample.c up-samples every component by (h_max / h_c, v_max / v_c) when these are integral, so a
  // 3-component frame of any such sampling (4:4:0, 4:1:1 too) has an RGB24 / YUV444 output
  plan->up_integral = true;
  for (int i = 0; i < ncomp; i++) {
    plan->up_h[i] = max_h % f.hs[i] == 0 ? max_h / f.hs[i] : 0;
    plan->up_v[i] = max_v % f.vs[i] == 0 ? max_v / f.vs[i] : 0;
    plan->up_integral = plan->up_integral && plan->up_h[i] && plan->up_v[i];
  }
  if ((flags & HCJ_FLAG_LIBJPEG) && ncomp == 3 && plan->up_integral) f.rgb_bytes = (size_t)f.width * f.height * 3;
  return HCJ_OK;
}

int build_lut(const hcj_dht &t, HuffLut *lut) {
  // Specification.create_code_table, tables.ml:27-45
  struct Code {
    int length, bits, data;
  };
  std::vector<Code> codes;
  int64_t code = 0;
  int data_pos = 0;
  for (int lp = 0; lp < 16; lp++) {
    if (t.lengths[lp] == 0) {
      code <<= 1;
    } else {
      for (int i = 0; i < t.lengths[lp]; i++) codes.push_back({lp + 1, (int)(code + i), t.values[data_pos + i]});
      code = (code + t.lengths[lp]) << 1;
      data_pos += t.lengths[lp];
    }
  }
  if (t.table_class == 0)
    for (const Code &c : codes)
      if (c.data > 15) return HCJ_ERR_UNSUPPORTED_GEOMETRY;  // stated domain limit (DC category)
  // Lut.create, tables.ml:490-501: later codes overwrite earlier ones
  int max_bits = 0;
  for (const Code &c : codes) max_bits = std::max(max_bits, c.length);
  lut->max_bits = max_bits;
  lut->full.assign((size_t)1 << max_bits, 0);
  for (const Code &c : codes) {
    int null_bits = max_bits - c.length;
    int64_t first = (int64_t)c.bits << null_bits, count = (int64_t)1 << null_bits;
    if (first + count > (int64_t)lut->full.size()) return HCJ_ERR_BAD_HUFFMAN_TABLE;
    for (int64_t i = first; i < first + count; i++) lut->full[i] = (uint16_t)((c.length << 8) | c.data);
  }
  // Primary table over the next HCJ_LUT_BITS bits: an entry is resolved here when every full-table
  // slot under the prefix agrees on a code no longer than the prefix.  Other prefixes get one of the
  // HCJ_LUT_NSUB sub-tables (a verbatim slice of the full table); if those run out the entry stays 0
  // and the kernels consult the full table in global memory.
  lut->primary.assign(HCJ_LUT_ENTRIES, 0);
  int nsub = 0;
  for (int p = 0; p < HCJ_LUT_SIZE; p++) {
    if (max_bits <= HCJ_LUT_BITS) {
      lut->primary[p] = lut->full[p >> (HCJ_LUT_BITS - max_bits)];
    } else {
      int sh = max_bits - HCJ_LUT_BITS;
      size_t n = (size_t)1 << sh, base = (size_t)p << sh;
      uint16_t e = lut->full[base];
      bool same = ((e >> 8) <= HCJ_LUT_BITS);
      bool any = e != 0;
      for (size_t i = 1; i < n; i++) {
        same = same && lut->full[base + i] == e;
        any = any || lut->full[base + i] != 0;
      }
      if (same) {
        lut->primary[p] = e;  // includes "all None" (0): the full-table lookup then finds None as well
      } else if (any && nsub < HCJ_LUT_NSUB && sh <= HCJ_LUT_SUB_BITS) {
        for (size_t i = 0; i < n; i++) lut->primary[HCJ_LUT_SIZE + nsub * HCJ_LUT_SUB_SIZE + i] = lut->full[base + i];
        lut->primary[p] = (uint16_t)(0x8000 | nsub);
        nsub++;
      } else {
        lut->primary[p] = 0;
      }
    }
  }
  return HCJ_OK;
}

// ---- encoder defaults (ITU-T T.81 Annex K; tables.ml:54-476, quant_tables.ml:3-137) -------------
namespace {
const uint8_t kDcLumaLengths[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
const uint8_t kDcChromaLengths[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
const uint8_t kDcValues[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
const uint8_t kAcLumaLengths[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
const uint8_t kAcChromaLengths[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
// Values in (run << 4 | size) form, listed per code length as in Annex K.5 / K.6.
const uint8_t kAcLumaValues[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
    0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
    0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
    0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
    0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
const uint8_t kAcChromaValues[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
    0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
    0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
    0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
    0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
    0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
// Annex K.1 / K.2 values as the model stores them (natural order, used as if zig-zag; SURVEY A.6).
const uint8_t kQuantLuma[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
const uint8_t kQuantChroma[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                  24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                                  99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                  99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
}  // namespace

void default_spec(int which, const uint8_t **lengths, const uint8_t **values, int *nvalues) {
  switch (which) {
    case 0: *lengths = kDcLumaLengths; *values = kDcValues; *nvalues = 12; break;
    case 1: *lengths = kDcChromaLengths; *values = kDcValues; *nvalues = 12; break;
    case 2: *lengths = kAcLumaLengths; *values = kAcLumaValues; *nvalues = 162; break;
    default: *lengths = kAcChromaLengths; *values = kAcChromaValues; *nvalues = 162; break;
  }
}

void quant_scale(bool chroma, int quality, uint16_t out[64]) {  // quant_tables.ml:139-147
  const uint8_t *table = chroma ? kQuantChroma : kQuantLuma;
  int q = std::min(100, std::max(1, quality));
  int s = q < 50 ? 5000 / q : 200 - 2 * q;
  for (int i = 0; i < 64; i++) {
    int d = (table[i] * s + 50) / 100;
    out[i] = (uint16_t)std::min(255, std::max(1, d));
  }
}

void encoder_tables(int which_dc, int which_ac, uint32_t dc[16], uint32_t ac[256]) {
  // Encoder.dc_table sorts the codes by category and indexes by size (tables.ml:505-514, encoder.ml:157);
  // Encoder.ac_table groups by run and indexes [run][size] (tables.ml:516-544, encoder.ml:164).  With
  // the default specs every category / run is present, so a direct [(run << 4) | size] map is the same.
  memset(dc, 0, sizeof(uint32_t) * 16);
  memset(ac, 0, sizeof(uint32_t) * 256);
  for (int pass = 0; pass < 2; pass++) {
    const uint8_t *lengths, *values;
    int nv;
    default_spec(pass == 0 ? which_dc : which_ac, &lengths, &values, &nv);
    uint32_t code = 0;
    int pos = 0;
    for (int lp = 0; lp < 16; lp++) {  // tables.ml:27-45
      for (int i = 0; i < lengths[lp]; i++) {
        uint32_t e = ((code + i) << 8) | (uint32_t)(lp + 1);
        if (pass == 0) dc[values[pos + i] & 15] = e;
        else ac[values[pos + i]] = e;
      }
      code = (code + lengths[lp]) << 1;
      pos += lengths[lp];
    }
  }
}

int plan_encode(int width, int height, int chroma, int quality, int restart_interval, EncodePlan *p) {
  memset(p, 0, sizeof(*p));
  static const int s420[6] = {2, 2, 1, 1, 1, 1}, s422[6] = {2, 2, 1, 2, 1, 2}, s444[6] = {1, 1, 1, 1, 1, 1};
  // encoder.ml:347-349; 400 = Parameters.monochrome (:351-368): one component, luma tables only
  const int *s = chroma == 420 ? s420 : chroma == 422 ? s422 : (chroma == 444 || chroma == 400) ? s444 : nullptr;
  if (!s || width < 1 || height < 1 || width > 65535 || height > 65535 || restart_interval < 0 || restart_interval > 65535)
    return HCJ_ERR_ENCODER_PARAMS;
  p->width = width;
  p->height = height;
  p->chroma = chroma;
  p->quality = quality;
  p->restart_interval = restart_interval;
  p->ncomp = chroma == 400 ? 1 : 3;
  quant_scale(false, quality, p->qt[0]);
  quant_scale(true, quality, p->qt[1]);
  int max_h = 0, max_v = 0;
  for (int i = 0; i < p->ncomp; i++) {
    p->hs[i] = s[2 * i];
    p->vs[i] = s[2 * i + 1];
    max_h = std::max(max_h, p->hs[i]);
    max_v = std::max(max_v, p->vs[i]);
  }
  int bpm = 0;
  for (int i = 0; i < p->ncomp; i++) {  // Encoder.create, encoder.ml:450-463
    int64_t w = (int64_t)width * p->hs[i] / max_h, h = (int64_t)height * p->vs[i] / max_v;
    p->plane_w[i] = (int)round_up(w, 8 * p->hs[i]);
    p->plane_h[i] = (int)round_up(h, 8 * p->vs[i]);
    p->src_w[i] = i == 0 ? width : (chroma == 444 ? width : width / 2);  // frame.ml:7-19
    p->src_h[i] = i == 0 ? height : (chroma == 420 ? height / 2 : height);
    for (int y = 0; y < p->vs[i]; y++)
      for (int x = 0; x < p->hs[i]; x++) {
        p->blk_comp[bpm] = i;
        p->blk_bx[bpm] = x;
        p->blk_by[bpm] = y;
        bpm++;
      }
  }
  p->bpm = bpm;
  p->mcus_wide = p->plane_w[0] / (8 * p->hs[0]);  // encoder.ml:477-480
  p->mcus_high = p->plane_h[0] / (8 * p->vs[0]);
  p->nblocks = (int64_t)p->mcus_wide * p->mcus_high * bpm;
  // bit offsets within a frame are 32-bit on the device: a block is at most 3456 bits (hcj_encode_bound)
  if (p->nblocks * 3456 >= ((int64_t)1 << 32)) return HCJ_ERR_UNSUPPORTED_GEOMETRY;
  // encode_block reads through a bounds-checked Plane (encoder.ml:85): per-component rounding can
  // disagree for odd sizes (SURVEY A.10) and the model raises.
  for (int i = 0; i < p->ncomp; i++)
    if (p->mcus_wide * p->hs[i] * 8 > p->plane_w[i] || p->mcus_high * p->vs[i] * 8 > p->plane_h[i])
      return HCJ_ERR_PLANE_BOUNDS;
  return HCJ_OK;
}

namespace {
void put16(std::vector<uint8_t> *o, int v) {
  o->push_back((uint8_t)(v >> 8));
  o->push_back((uint8_t)v);
}
void marker(std::vector<uint8_t> *o, int code) {  // encoder.ml:207-210
  o->push_back(0xff);
  o->push_back((uint8_t)code);
}
}  // namespace

void write_headers(const EncodePlan &p, std::vector<uint8_t> *o) {  // encoder.ml:371-418
  marker(o, SOI);
  static const char tag[] = "Hardcaml JPEG.";  // write_app0, encoder.ml:231-237,383
  marker(o, APP0);
  put16(o, 2 + (int)strlen(tag));
  o->insert(o->end(), tag, tag + strlen(tag));
  const int ntab = p.ncomp == 1 ? 1 : 2;  // Parameters.monochrome carries one table of each kind (encoder.ml:351-368)
  for (int t = 0; t < ntab; t++) {  // write_dqt + Dqt.encode, markers.ml:170-183
    marker(o, DQT);
    put16(o, 3 + 64);
    o->push_back((uint8_t)t);  // Pq = 0, Tq = t
    for (int i = 0; i < 64; i++) o->push_back((uint8_t)p.qt[t][i]);
  }
  marker(o, SOF0);  // write_sof + Sof.encode, markers.ml:61-71
  put16(o, 2 + 6 + p.ncomp * 3);
  o->push_back(8);
  put16(o, p.height);
  put16(o, p.width);
  o->push_back((uint8_t)p.ncomp);
  for (int i = 0; i < p.ncomp; i++) {
    o->push_back((uint8_t)(i + 1));
    o->push_back((uint8_t)((p.hs[i] << 4) | p.vs[i]));
    o->push_back((uint8_t)(i ? 1 : 0));
  }
  for (int cls = 0; cls < 2; cls++)  // dc 0, dc 1, ac 0, ac 1 (encoder.ml:405-408)
    for (int t = 0; t < ntab; t++) {
      const uint8_t *lengths, *values;
      int nv;
      default_spec(cls * 2 + t, &lengths, &values, &nv);
      marker(o, DHT);  // Dht.encode, markers.ml:222-231
      put16(o, 3 + 16 + nv);
      o->push_back((uint8_t)((cls << 4) | t));
      o->insert(o->end(), lengths, lengths + 16);
      o->insert(o->end(), values, values + nv);
    }
  if (p.restart_interval > 0) {  // stated extension
    marker(o, DRI);
    put16(o, 4);
    put16(o, p.restart_interval);
  }
  marker(o, SOS);  // write_sos + Sos.encode, markers.ml:131-150
  put16(o, 2 + 4 + p.ncomp * 2);
  o->push_back((uint8_t)p.ncomp);
  for (int i = 0; i < p.ncomp; i++) {
    o->push_back((uint8_t)(i + 1));
    o->push_back((uint8_t)(i ? 0x11 : 0x00));
  }
  o->push_back(0);
  o->push_back(63);
  o->push_back(0);
}

}  // namespace hcj
