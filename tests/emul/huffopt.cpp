// huffopt.cpp — TEST INFRASTRUCTURE: the optimal-table logic of HCJ_ENC_OPTIMIZE_HUFFMAN (hcj_device.cuh) compiled with
// g++: the serial gen_optimal_table, k2_optimal_table driven by a single lane, and block_symbols_sparse beside
// encode_block_fields_sparse.  Nothing in the product links or calls this file.
#include <stdint.h>

#include "hcj_device.cuh"

using namespace hcjdev;

extern "C" {

int emu_gen_optimal_table(const uint32_t *freq /* [256] */, uint8_t *bits, uint8_t *huffval) {
  uint32_t f[257];
  for (int i = 0; i < 256; i++) f[i] = freq[i];
  f[256] = 1;
  return gen_optimal_table(f, bits, huffval);
}

int emu_k2_single_lane(const uint32_t *freq /* [256] */, uint8_t *bits, uint8_t *huffval) {
  static K2Scratch s;
  const K2Lanes w{0, 1};
  return k2_optimal_table(w, freq, s, bits, huffval);
}

// canonical codes of (bits, huffval) in the kernels' format: codes[256] (dc: indexed by symbol & 15)
void emu_canonical_codes(const uint8_t *bits, const uint8_t *huffval, int dc, uint32_t *codes) {
  canonical_codes(bits, huffval, dc != 0, codes);
}

// One block (64 zig-zag coefficients, DC slot ignored) with DC difference dcdiff.  visited[]: (is_ac << 8) | symbol of
// every block_symbols_sparse visit; emitted[]: the same for every code encode_block_fields_sparse emits, read back from
// tables whose code for a symbol is that 9-bit value.  Returns (number visited) | (number emitted) << 16, or -1 when
// the two walks disagree on success.
int64_t emu_block_symbols(const int16_t *blk, int32_t dcdiff, uint32_t *visited, uint32_t *emitted) {
  uint64_t nz = 0;
  for (int k = 0; k < 64; k++) nz |= (uint64_t)(blk[k] != 0) << k;
  auto coef = [blk](int k) { return (int32_t)blk[k]; };
  int nv = 0, ne = 0;
  auto visit = [&](bool is_ac, uint32_t sym) { visited[nv++] = (is_ac ? 256u : 0u) | sym; };
  const bool ok1 = block_symbols_sparse(nz, coef, dcdiff, visit);
  uint32_t dc[16], ac[256];
  for (uint32_t i = 0; i < 16; i++) dc[i] = (i << 8) | 9u;
  for (uint32_t i = 0; i < 256; i++) ac[i] = ((256u | i) << 8) | 9u;
  auto emit = [&](uint32_t bits, uint32_t n) {  // every field starts with a 9-bit code
    if (n >= 9) emitted[ne++] = bits >> (n - 9);
  };
  const bool ok2 = encode_block_fields_sparse(nz, coef, dcdiff, dc, ac, emit);
  if (ok1 != ok2) return -1;
  return (int64_t)nv | ((int64_t)ne << 16);
}

}  // extern "C"
