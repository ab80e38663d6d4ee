// scaled.cpp — TEST INFRASTRUCTURE: the scaled decode's per-thread transforms (reconstruct_scaled in hcj_device.cuh)
// compiled with g++ and driven block by block, like emul.cpp drives the other device logic.  Nothing in the product
// links or calls this file.
#include <stdint.h>

#include "hcj_device.cuh"

using namespace hcjdev;

extern "C" {

// n zig-zag int16 blocks (DC absolute) with one zig-zag quant table -> n blocks of k x k samples.
// wide < 0: the path the IDCT kernel takes (64-bit column pass when some quant entry exceeds 255 or the block's
// sum(|dequantised coefficient|) reaches HCJ_IDCT_L1_LIMIT, i.e. when the entropy decoders flag it); 0 / 1 force the
// 32-bit / 64-bit column pass.
void emu_reconstruct_scaled(const int16_t *coefs, int64_t n, const uint16_t *qt, int k, int wide, uint8_t *out) {
  int32_t q[64];
  bool table_wide = false;
  for (int i = 0; i < 64; i++) {
    q[i] = qt[i];
    table_wide |= qt[i] > 255;
  }
  for (int64_t b = 0; b < n; b++) {
    const int16_t *c = coefs + b * 64;
    uint32_t cw[32], pix[4];
    uint64_t l1 = 0;
    for (int j = 0; j < 32; j++) cw[j] = (uint32_t)(uint16_t)c[2 * j] | ((uint32_t)(uint16_t)c[2 * j + 1] << 16);
    for (int i = 0; i < 64; i++) l1 += (uint64_t)(c[i] < 0 ? -(int64_t)c[i] : c[i]) * (uint64_t)qt[i];
    const bool w = wide < 0 ? (table_wide || l1 >= (uint64_t)HCJ_IDCT_L1_LIMIT) : wide != 0;
    reconstruct_scaled(cw, q, k, w, pix);
    for (int r = 0; r < k; r++)
      for (int i = 0; i < k; i++) out[(b * k + r) * k + i] = (uint8_t)(pix[r] >> (8 * i));
  }
}

int emu_scaled_l1_limit() { return HCJ_IDCT_L1_LIMIT; }

}  // extern "C"
