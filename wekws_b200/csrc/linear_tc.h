// Kernel argument block of the tensor-core dense Linear (linear_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace wekws {

struct LinearTcArgs {
  const float* x;          // (rows, K) fp32, row stride x_stride floats (16-byte aligned rows)
  float* out;              // (rows, N) fp32, row stride out_stride floats
  const uint8_t* wimg;     // [n tile of 128][K slab of 64] bf16 hi|lo images, 32 KB each (linear_tc_pack)
  const float* bias;       // N floats, padded to a multiple of 128
  long long rows, x_stride, out_stride;
  int N, K, act;
  int n_mtiles;            // set by linear_tc_launch
};

size_t linear_tc_image_bytes(int N, int K);
bool linear_tc_eligible(int N, int K);
// wt: W^T as [K][ldn] floats (ldn >= N); writes linear_tc_image_bytes(N, K) bytes
void linear_tc_pack(uint8_t* dst, const float* wt, int ldn, int N, int K);
int linear_tc_launch(LinearTcArgs a, cudaStream_t st);

}  // namespace wekws
