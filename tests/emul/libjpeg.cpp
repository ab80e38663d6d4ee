// libjpeg.cpp — TEST INFRASTRUCTURE: the HCJ_FLAG_LIBJPEG per-thread functions of hcj_device.cuh (islow_fast / islow_wide,
// libjpeg_upsample) compiled with g++ and driven block by block and sample by sample.  Nothing in the product links or
// calls this file.
#include <stdint.h>

#include "hcj_device.cuh"

using namespace hcjdev;

extern "C" {

// n zig-zag int16 blocks (DC absolute) with one zig-zag quant table -> n blocks of 8 x 8 samples.
// wide < 0: the path the IDCT kernel takes (64-bit column pass when some quant entry exceeds 255 or the block's
// sum(|dequantised coefficient|) reaches HCJ_IDCT_L1_LIMIT, i.e. when the entropy decoders flag it); 0 / 1 force the
// 32-bit / 64-bit column pass.
void emu_islow(const int16_t *coefs, int64_t n, const uint16_t *qt, int wide, uint8_t *out) {
  int32_t q[64], qd[64];
  bool table_wide = false;
  for (int i = 0; i < 64; i++) {
    q[i] = qt[i];
    qd[i] = HCJ_QD(i, qt[i] & 0xff);
    table_wide |= qt[i] > 255;
  }
  for (int64_t b = 0; b < n; b++) {
    const int16_t *c = coefs + b * 64;
    uint32_t cw[32], pix[16];
    uint64_t l1 = 0;
    for (int j = 0; j < 32; j++) cw[j] = (uint32_t)(uint16_t)c[2 * j] | ((uint32_t)(uint16_t)c[2 * j + 1] << 16);
    for (int i = 0; i < 64; i++) l1 += (uint64_t)(c[i] < 0 ? -(int64_t)c[i] : c[i]) * (uint64_t)qt[i];
    const bool w = wide < 0 ? (table_wide || l1 >= (uint64_t)HCJ_IDCT_L1_LIMIT) : wide != 0;
    if (w) islow_wide(cw, q, pix);
    else islow_fast(cw, qd, pix);
    for (int k = 0; k < 64; k++) out[b * 64 + k] = (uint8_t)(pix[k >> 2] >> (8 * (k & 3)));
  }
}

// One component up-sampled to W x H (out: W * H bytes) from its plane (pitch bytes per row, rw x rh real samples).
void emu_upsample(const uint8_t *plane, int pitch, int rw, int rh, int hr, int vr, int W, int H, uint8_t *out) {
  for (int y = 0; y < H; y++)
    for (int x = 0; x < W; x++) out[(int64_t)y * W + x] = (uint8_t)libjpeg_upsample(plane, pitch, rw, rh, hr, vr, x, y);
}

int emu_islow_l1_limit() { return HCJ_IDCT_L1_LIMIT; }

}  // extern "C"
