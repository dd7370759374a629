// Dense Linear on tcgen05 for wide outputs: Y[rows][N] = act(X[rows][K] . W[N][K]^T + b), K <= 256, any N.
// Used for the CTC classifier heads (classifier.py:63-67 with output_dim 2599, examples/hi_xiaowen/s0/conf/
// ds_tcn_ctc.yaml:31-42) behind the tensor-core DS-TCN backbone: at odim 2599 the classifier is 1.33 MFLOP per frame,
// 2.3x the whole backbone, and used to force the model onto the FP32 kernel.
//
// bf16 x3 operand split, fp32 accumulate (same arithmetic as the backbone kernels).  One CTA per 128-row tile
// (persistent over tiles):
//   * the tile's A operand (128 rows x K, hi | lo) is written to TENSOR MEMORY once per tile by the row-owner threads
//     (global fp32 row -> split -> tcgen05.st) and reused for every output tile;
//   * W streams from L2 as pre-swizzled K-major SWIZZLE_128B images (128 output columns x 64 K, hi | lo = 32 KB,
//     the format of dstcn_tc.cu) through a 4-slot cp.async.bulk ring;
//   * per output tile of 128 columns: K/64 slabs x 3 passes x 4 MMAs (M = 128, N = 128, K = 16) into one of two TMEM
//     accumulators, so the epilogue (tcgen05.ld, bias, activation, 512 contiguous bytes per row to global) of tile
//     n overlaps the MMAs of tile n + 1.
// Warps: 0-3 row owners (operand + epilogue), 4 MMA issuer, 5 weight loader.
#include <string.h>

#include "common.cuh"
#include "linear_tc.h"
#include "tc_common.cuh"
#include "tc_pack.h"

namespace wekws {
namespace {

using namespace tc;

constexpr int NT = 192;
constexpr int W_SLOT = 32768, NW = 4;
constexpr int SMEM_BYTES = NW * W_SLOT + 1024;
constexpr int TM_AHI = 0, TM_ALO = 128, TM_D = 256, TM_COLS = 512;
constexpr int NTILE = 128;     // output columns per accumulator

__global__ void __launch_bounds__(NT, 1) linear_tc_kernel(const LinearTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  __shared__ uint64_t w_bar[NW], w_free[NW], d_full[2], d_free[2], a_rdy, a_free;
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

  if (tid == 0) {
    for (int i = 0; i < NW; ++i) { mbar_init(&w_bar[i], 1); mbar_init(&w_free[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&d_full[i], 1); mbar_init(&d_free[i], 4); }
    mbar_init(&a_rdy, 4);
    mbar_init(&a_free, 1);
    mbar_fence_init();
  }
  if (warp == 4) tmem_alloc(&tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform32(tmem_slot);      // warp-uniform: MMA operands are then built in uniform registers
  const int nslab = a.K / 64, ntn = (a.N + NTILE - 1) / NTILE;
  const int my_tiles = a.n_mtiles > (int)blockIdx.x ? (a.n_mtiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t idesc = make_idesc_bf16(128, NTILE);

  if (warp < 4) {
    // ================================================================== ROW OWNERS: operand rows, then epilogues
    const int row = 32 * warp + lane;
    const uint32_t trow = tmem + ((uint32_t)(32 * warp) << 16);
    uint32_t dfull_par = 0, afree_par = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const long long r = (long long)(blockIdx.x + it * gridDim.x) * 128 + row;
      const bool live = r < a.rows;
      if (it > 0) {                                    // the previous tile's MMAs have read the operand
        mbar_wait(&a_free, afree_par);
        afree_par ^= 1;
        tc_fence_after();
      }
      const float4* src = reinterpret_cast<const float4*>(a.x + r * a.x_stride);
      for (int c0 = 0; c0 < a.K / 8; c0 += 8) {        // 8 chunks of 8 values (16 float4) in flight
        float4 v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = (live && 2 * c0 + i < a.K / 4) ? __ldg(src + 2 * c0 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          if (c0 + c < a.K / 8) {
            uint32_t h[4], l[4];
            split2(v[2 * c].x, v[2 * c].y, h[0], l[0]); split2(v[2 * c].z, v[2 * c].w, h[1], l[1]);
            split2(v[2 * c + 1].x, v[2 * c + 1].y, h[2], l[2]); split2(v[2 * c + 1].z, v[2 * c + 1].w, h[3], l[3]);
            tmem_st4(trow + TM_AHI + 4 * (c0 + c), h);
            tmem_st4(trow + TM_ALO + 4 * (c0 + c), l);
          }
        }
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&a_rdy);
      float* orow = a.out + r * a.out_stride;
      for (int n = 0; n < ntn; ++n) {
        const int buf = n & 1;
        mbar_wait(&d_full[buf], (dfull_par >> buf) & 1);
        dfull_par ^= 1u << buf;
        tc_fence_after();
        const int n0 = n * NTILE;
#pragma unroll 1
        for (int q = 0; q < 4; ++q) {                  // 32 columns at a time
          uint32_t d[32];
          tmem_ld32_nowait(trow + TM_D + NTILE * buf + 32 * q, d);
          tmem_ld_wait();
          if (q == 3) {                                // this warp is done with the accumulator
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&d_free[buf]);
          }
          if (!live) continue;
          const int c0 = n0 + 32 * q;
          if (c0 + 32 <= a.N && (a.out_stride & 3) == 0) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(a.bias + c0) + j);
              float4 y = make_float4(__uint_as_float(d[4 * j]) + b.x, __uint_as_float(d[4 * j + 1]) + b.y,
                                     __uint_as_float(d[4 * j + 2]) + b.z, __uint_as_float(d[4 * j + 3]) + b.w);
              if (a.act == WEKWS_ACT_SIGMOID) { y.x = sigmoidf_acc(y.x); y.y = sigmoidf_acc(y.y); y.z = sigmoidf_acc(y.z); y.w = sigmoidf_acc(y.w); }
              *reinterpret_cast<float4*>(orow + c0 + 4 * j) = y;
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              if (c0 + j < a.N) {
                float y = __uint_as_float(d[j]) + __ldg(a.bias + c0 + j);
                if (a.act == WEKWS_ACT_SIGMOID) y = sigmoidf_acc(y);
                orow[c0 + j] = y;
              }
            }
          }
        }
      }
    }
  } else if (warp == 4) {
    // ================================================================== MMA ISSUER (whole warp, tcgen05 instructions elected:
    // uniform values keep the descriptors in uniform registers, see tc_common.cuh elect_one_sync)
    {
      uint32_t seq = 0, ardy_par = 0, dfree_par = 0, used[2] = {0, 0};
      for (int it = 0; it < my_tiles; ++it) {
        mbar_wait(&a_rdy, ardy_par);
        ardy_par ^= 1;
        tc_fence_after();
        for (int n = 0; n < ntn; ++n) {
          const int buf = n & 1;
          if (used[buf]) {                             // the epilogue has drained this accumulator
            mbar_wait(&d_free[buf], (dfree_par >> buf) & 1);
            dfree_par ^= 1u << buf;
            tc_fence_after();
          }
          used[buf] = 1;
          const uint32_t d = tmem + TM_D + NTILE * buf;
          uint32_t acc = 0;
          for (int s = 0; s < nslab; ++s, ++seq) {
            const uint32_t slot = seq % NW;
            mbar_wait(&w_bar[slot], (seq / NW) & 1);
            tc_fence_after();
            const uint64_t whi = make_sdesc_sw128(smem_u32(base + slot * W_SLOT)), wlo = make_sdesc_sw128(smem_u32(base + slot * W_SLOT) + 16384);
            const uint32_t ahi = tmem + TM_AHI + 32 * s, alo = tmem + TM_ALO + 32 * s;
            if (elect_one_sync()) {
              for (int k = 0; k < 4; ++k) umma_bf16_ts(d, ahi + 8 * k, whi + 2 * k, idesc, k == 0 ? acc : 1u);
              for (int k = 0; k < 4; ++k) umma_bf16_ts(d, alo + 8 * k, whi + 2 * k, idesc, 1);
              for (int k = 0; k < 4; ++k) umma_bf16_ts(d, ahi + 8 * k, wlo + 2 * k, idesc, 1);
              umma_commit(&w_free[slot]);
            }
            acc = 1;
          }
          if (elect_one_sync()) umma_commit(&d_full[buf]);
        }
        if (elect_one_sync()) umma_commit(&a_free);
      }
    }
  } else {
    // ================================================================== WEIGHT LOADER (lane 0): images [n tile][slab]
    if (lane == 0) {
      const uint32_t total = (uint32_t)my_tiles * (uint32_t)ntn * (uint32_t)nslab, per = (uint32_t)ntn * (uint32_t)nslab;
      for (uint32_t seq = 0; seq < total; ++seq) {
        const uint32_t slot = seq % NW;
        if (seq >= NW) mbar_wait_backoff(&w_free[slot], ((seq / NW) - 1) & 1);
        mbar_arrive_expect_tx(&w_bar[slot], W_SLOT);
        bulk_g2s(base + slot * W_SLOT, a.wimg + (size_t)(seq % per) * W_SLOT, W_SLOT, &w_bar[slot]);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

size_t linear_tc_image_bytes(int N, int K) { return (size_t)((N + NTILE - 1) / NTILE) * (size_t)(K / 64) * W_SLOT; }
bool linear_tc_eligible(int N, int K) { return K >= 64 && K <= 256 && K % 64 == 0 && N >= 1; }

void linear_tc_pack(uint8_t* dst, const float* wt, int ldn, int N, int K) {
  const int ntn = (N + NTILE - 1) / NTILE, nslab = K / 64;
  memset(dst, 0, (size_t)ntn * nslab * W_SLOT);          // rows beyond N stay zero
  for (int nt = 0; nt < ntn; ++nt)
    for (int s = 0; s < nslab; ++s) {
      const int rows = N - nt * NTILE < NTILE ? N - nt * NTILE : NTILE;
      write_sw128_image(dst + (size_t)(nt * nslab + s) * W_SLOT, 16384, wt + (size_t)(64 * s) * ldn + nt * NTILE, rows,
                        1, (size_t)ldn, 64);
    }
}

int linear_tc_launch(LinearTcArgs a, cudaStream_t st) {
  WEKWS_REQUIRE(a.rows >= 1 && linear_tc_eligible(a.N, a.K), "linear_tc_launch: unsupported shape (rows %lld, N %d, K %d)",
                (long long)a.rows, a.N, a.K);
  WEKWS_REQUIRE(((uintptr_t)a.x & 15) == 0 && (a.x_stride & 3) == 0, "linear_tc_launch: input rows must be 16-byte aligned");
  a.n_mtiles = (int)((a.rows + 127) / 128);
  static bool attr_set[64] = {false};
  if (int rc = set_max_dynamic_smem_once(attr_set, SMEM_BYTES, linear_tc_kernel)) return rc;
  const int sms = device_sm_count();
  const int grid = a.n_mtiles < sms ? a.n_mtiles : sms;
  linear_tc_kernel<<<grid, NT, SMEM_BYTES, st>>>(a);
  return check_launch("linear_tc_kernel");
}

}  // namespace wekws
