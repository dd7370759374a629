// Host-side packing of the bf16 x3 weight images the tcgen05 kernels read (mdtc_tc.cu, tcn_tc.cu, dstcn_tc.cu,
// linear_tc.cu, gru_tc.cu): every weight w is stored as hi = bf16(w) and lo = bf16(w - hi).
#pragma once
#include <stddef.h>
#include <stdint.h>
#include <string.h>

namespace wekws {

// round-to-nearest-even fp32 -> bf16 (as __floats2bfloat162_rn does on the device)
inline uint16_t bf16_rn(float x) {
  uint32_t u;
  memcpy(&u, &x, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);      // inf / nan
  u += 0x7FFFu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

inline float bf16_to_f(uint16_t h) {
  uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// K-major SWIZZLE_128B image of `rows` x 64 K (tc_common.cuh layout: row n at n * 128 bytes, its 16-byte chunk c at
// chunk c ^ (n & 7)), hi at dst and lo at dst + lo_off.  Element (n, k) is src[n * n_stride + k * k_stride] for k < kn
// and zero for kn <= k < 64.
inline void write_sw128_image(uint8_t* dst, size_t lo_off, const float* src, int rows, size_t n_stride, size_t k_stride,
                              int kn) {
  for (int n = 0; n < rows; ++n)
    for (int kk = 0; kk < 64; ++kk) {
      const float w = kk < kn ? src[(size_t)n * n_stride + (size_t)kk * k_stride] : 0.f;
      const uint16_t hi = bf16_rn(w), lo = bf16_rn(w - bf16_to_f(hi));
      const size_t off = (size_t)n * 128 + (size_t)(((kk >> 3) ^ (n & 7)) << 4) + (size_t)(kk & 7) * 2;
      memcpy(dst + off, &hi, 2);
      memcpy(dst + lo_off + off, &lo, 2);
    }
}

}  // namespace wekws
