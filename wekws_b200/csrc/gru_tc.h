// Kernel argument block of the tensor-core (weight-streaming) GRU kernel (gru_tc.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace wekws {

struct GruTcArgs {
  const float* feats;      // (B, T, idim)
  const float* in_cache;   // (L, B, H) or nullptr (== zeros)
  float* out;              // (B, T, odim)
  float* out_cache;        // (L, B, H)
  const float* vec;        // same fp32 blob as the FP32 kernel (pack_gru): CMVN, biases, classifier
  const uint8_t* wimg;     // per-step weight stream: 16 KB bf16 hi|lo operand chunks in consumption order (gru_tc_pack)
  int B, T, L, idim, odim, act, has_cmvn;
  int v_mean, v_istd, v_bp, v_layers, v_layer_stride, v_wc, v_bc;
  int n_tiles;
  int ms;                  // streams per CTA tile: 16, 32 or 64 (set by gru_tc_launch)
};

size_t gru_tc_image_bytes(int L, int idim);
bool gru_tc_eligible(int L, int H, int idim);
void gru_tc_pack(uint8_t* dst, const float* wp, int idim, const float* const* wih, const float* const* whh, int L);
int gru_tc_launch(GruTcArgs a, cudaStream_t st);

}  // namespace wekws
