// Tensor-core GRU forward with weight streaming (KWSModel.forward with the GRU backbone, kws_model.py:128-133; PyTorch
// gate order r, z, n -- see gru.cu for the FP32 kernel of the same math).
//
// Shape of the problem at the streaming operating point (B = 512 streams, one frame per call): 0.2 GFLOP against 786 KB
// of weights.  The FP32 kernel spreads the streams over all 148 SMs, so every SM pulls all weights out of L2 for 3-4
// streams: 116 MB of L2 egress and ~20 us per step, and its FMA loop is bound by shared-memory operand loads.  Here a
// CTA owns a tile of 64 streams and the GEMMs are TRANSPOSED: D^T[gate row][stream] = W[gate row][k] * X^T[k][stream],
// i.e. the weights are the M = 128 operand (one gate of all 128 hidden units per MMA row block, streamed from L2 through
// a ring of 16 KB pre-swizzled bf16 hi|lo chunks by bulk async copies), the activations are the N = 64 operand (K-major
// SWIZZLE_128B images in shared memory: features, x0, h of each layer, each split into bf16 hi + lo once by its producer)
// and the accumulators put the hidden UNITS on the 128 TMEM lanes -- so the gate math runs on all four SM sub-partitions
// with one thread per (unit, 32 streams), the old h stays in fp32 registers for the whole call, and no CTA ever talks to
// another one.  fp32 parity through the bf16 x3 split (W_hi X_hi + W_hi X_lo + W_lo X_hi, fp32 accumulate).
//
// Per step and CTA: (2 ceil(idim/64) + 24 L) weight chunks = 786 KB for the shipped model, ~300 MMAs (M128 N64 K16),
// TMEM: layer l accumulators at columns [256 l, 256 l + 256) = r | z | n_x | n_h (64 streams each); the preprocessing
// Linear borrows layer 0's n_h block.  Measured dead end this replaces: hidden units split over an 8-CTA cluster with
// resident weights and DSMEM exchange of h -- three cluster barriers per step made it slower than the FP32 kernel
// (profiles/r02_gru_notes.md).
//
// Warps (384 threads): 0-7 unit owners (TMEM lane quadrant w % 4, stream half w / 4): epilogues, gate math, classifier,
// cache I/O; 8 MMA issue (one lane); 9 weight ring (one lane); 10-11 feature rows -> operand image for the next step.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "gru_tc.h"
#include "tc_common.cuh"
#include "tc_pack.h"

namespace wekws {
namespace {

using namespace tc;

constexpr int M = 64;                   // streams per CTA tile (the MMA N)
constexpr int H = 128;                  // hidden units (the MMA M)
constexpr int NT = 384;
constexpr int SLAB = M * 128;           // one activation K-slab image (64 rows x 128 B), 8 KB
constexpr int IMG = 4 * SLAB;           // activation image: [slab 0 hi][slab 0 lo][slab 1 hi][slab 1 lo]
constexpr int CHUNK = H * 128;          // one weight chunk: 128 gate rows x 64 K, bf16, 16 KB
constexpr int NSLOT = 5;
// shared memory map (bytes, 1024-aligned)
constexpr int OFF_F = 0;                // feature image (K = idim <= 128)
constexpr int OFF_X0 = OFF_F + IMG;     // x0 = relu(Linear)
constexpr int OFF_H = OFF_X0 + IMG;     // h of layer l at OFF_H + l * IMG
constexpr int OFF_RING = OFF_H + 2 * IMG;
constexpr int OFF_END = OFF_RING + NSLOT * CHUNK;
constexpr int SMEM_BYTES = OFF_END + 1024;
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
constexpr int TM_COLS = 512;
constexpr int TM_R = 0, TM_Z = 64, TM_NX = 128, TM_NH = 192, TM_LAYER = 256, TM_LIN = TM_NH;

// byte offset of K element k (0..127) of stream row m inside an activation image (hi; lo at + SLAB)
__device__ __forceinline__ uint32_t a_off(int m, int k) {
  return (uint32_t)((k >> 6) * 2 * SLAB + m * 128 + ((((k & 63) >> 3) ^ (m & 7)) << 4) + (k & 7) * 2);
}
__device__ __forceinline__ void split1(float x, uint16_t& hi, uint16_t& lo) {
  const __nv_bfloat16 h = __float2bfloat16_rn(x);
  const __nv_bfloat16 l = __float2bfloat16_rn(x - __bfloat162float(h));
  hi = *reinterpret_cast<const uint16_t*>(&h);
  lo = *reinterpret_cast<const uint16_t*>(&l);
}
// Gates on the SFU approximations (ex2.approx, rcp.approx: ~1 ulp each): absolute error ~1e-7, far inside the
// fp32-parity budget (posterior 1e-4), and ~25 instructions per (unit, stream) instead of ~80 with expf / tanhf / IEEE
// division -- the gate math is on the critical path of every step.
__device__ __forceinline__ float ex2_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float LOG2E = 1.4426950408889634f;
// sigmoid(g + b) with nb = -b * log2(e) folded by the caller: 1 / (1 + 2^(-(g + b) log2 e))
__device__ __forceinline__ float sigmoid_fast(float g, float nb) { return rcp_fast(1.f + ex2_fast(fmaf(g, -LOG2E, nb))); }
// tanh(t) = 1 - 2 / (1 + 2^(2 t log2 e)); the exponent is clamped so that 2^x stays finite (tanh is 1 there anyway)
__device__ __forceinline__ float tanh_fast(float t) {
  return fmaf(-2.f, rcp_fast(1.f + ex2_fast(fminf(t * (2.f * LOG2E), 126.f))), 1.f);
}

struct Bars {
  uint64_t w_full[NSLOT], w_free[NSLOT];
  uint64_t f_rdy, lin_bar, x0_rdy, d_bar[2], h_rdy[2];
};

__device__ __forceinline__ void wait_flip(uint64_t* bar, uint32_t& par) {
  mbar_wait(bar, par);
  par ^= 1;
}
#ifndef GRU_TIMING
#define GRU_TIMING 0
#endif
#if GRU_TIMING
#define TWAIT(acc, stmt) { const long long t0_ = clock64(); stmt; acc += clock64() - t0_; }
#define TSEG_BEGIN(v) const long long v = clock64();
#define TSEG_END(acc, v) acc += clock64() - v;
#else
#define TWAIT(acc, stmt) { stmt; }
#define TSEG_BEGIN(v)
#define TSEG_END(acc, v)
#endif

// -------------------------------------------------------------------------------------------------- MMA issue (one lane)
// Measured on B200 (tests/native/mma_rate_probe.cu): one thread dispatches an M128 x N<=96 x K16 MMA every ~55 cycles at
// best (N = 128: 64, N = 256: 128 cycles), and only if the issue loop is a straight line of MMAs -- building a
// descriptor per instruction doubles that.  So everything below is unrolled over precomputed 64-bit descriptors.
struct Issuer {
  Bars* b;
  uint32_t idesc;
  uint64_t wdesc0;                         // descriptor of ring slot 0 (slot s: + s * CHUNK / 16 in the address field)
  uint32_t slot, full_par;                 // ring position (full_par: bit s = parity of the next fill of slot s)
  long long t_w;
  __device__ __forceinline__ uint64_t take() {             // wait for the next chunk, return its descriptor
    TWAIT(t_w, mbar_wait(&b->w_full[slot], (full_par >> slot) & 1u));
    tc_fence_after();
    return wdesc0 + (uint64_t)(slot * (CHUNK >> 4));
  }
  __device__ __forceinline__ void release() {              // the chunk's MMAs are issued: free its slot when they finish
    if (elect_one_sync()) umma_commit(&b->w_free[slot]);
    full_par ^= 1u << slot;
    slot = slot + 1 == NSLOT ? 0 : slot + 1;
  }
  // one K slab with `ksteps` MMA K steps: D (+)= W[:, slab] X[:, slab]^T with the x3 split
  __device__ __forceinline__ void slab_rt(uint32_t d, uint64_t xhi, int ksteps, uint32_t& acc) {
    const uint64_t xlo = xhi + (SLAB >> 4);
    const uint64_t whi = take();
    if (elect_one_sync()) {
      for (int k = 0; k < ksteps; ++k) umma_bf16(d, whi + 2 * k, xhi + 2 * k, idesc, k == 0 ? acc : 1u);
      for (int k = 0; k < ksteps; ++k) umma_bf16(d, whi + 2 * k, xlo + 2 * k, idesc, 1);
    }
    acc = 1;
    release();
    const uint64_t wlo = take();
    if (elect_one_sync()) {
      for (int k = 0; k < ksteps; ++k) umma_bf16(d, wlo + 2 * k, xhi + 2 * k, idesc, 1);
    }
    release();
  }
  // one gate block over K = 128 (two slabs of 4 K steps), fully unrolled; FRESH: the first MMA overwrites D
  template <bool FRESH>
  __device__ __forceinline__ void gate(uint32_t d, uint64_t ximg) {
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const uint64_t xhi = ximg + (uint64_t)(s * (2 * SLAB >> 4)), xlo = xhi + (SLAB >> 4);
      const uint64_t whi = take();
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d, whi + 2 * k, xhi + 2 * k, idesc, (FRESH && s == 0 && k == 0) ? 0u : 1u);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d, whi + 2 * k, xlo + 2 * k, idesc, 1u);
      }
      release();
      const uint64_t wlo = take();
      if (elect_one_sync()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_bf16(d, wlo + 2 * k, xhi + 2 * k, idesc, 1u);
      }
      release();
    }
  }
};

// executed by ALL lanes of the issue warp (uniform control flow and values); the MMAs / commits are elected
__device__ __noinline__ void issuer_role(const GruTcArgs& a, Bars* b_, uint32_t sbase_, uint32_t tmem_, int my_tiles_) {
  const uint32_t sbase = uniform32(sbase_), tmem = uniform32(tmem_);
  const int my_tiles = (int)uniform32((uint32_t)my_tiles_);
  const int L = (int)uniform32((uint32_t)a.L), T = (int)uniform32((uint32_t)a.T), idim = (int)uniform32((uint32_t)a.idim);
  Bars* b = reinterpret_cast<Bars*>(__cvta_shared_to_generic(uniform32(smem_u32(b_))));
  Issuer is{b, make_idesc_bf16(H, M), make_sdesc_sw128(sbase + OFF_RING), 0u, 0u, 0};
  long long t_f = 0, t_x0 = 0, t_h0 = 0, t_h1 = 0;
  const long long t_begin = clock64();
  uint32_t p_f = 0, p_x0 = 0, p_h0 = 0, p_h1 = 0;
  const int nsf = (idim + 63) >> 6;
  const uint64_t f_img = make_sdesc_sw128(sbase + OFF_F), x0_img = make_sdesc_sw128(sbase + OFF_X0);
  const uint64_t h0_img = make_sdesc_sw128(sbase + OFF_H), h1_img = make_sdesc_sw128(sbase + OFF_H + IMG);
  const uint32_t d0 = tmem, d1 = tmem + TM_LAYER;
  for (int it = 0; it < my_tiles; ++it) {
    wait_flip(&b->h_rdy[0], p_h0);                       // initial h images of the tile
    if (L == 2) wait_flip(&b->h_rdy[1], p_h1);
    for (int t = 0; t < T; ++t) {
      // ---- preprocessing Linear (subsampling.py:53-57): D_lin = Wp F^T
      TWAIT(t_f, wait_flip(&b->f_rdy, p_f));
      tc_fence_after();
      {
        uint32_t acc = 0;
        for (int s = 0; s < nsf; ++s) {
          const int rem = idim - 64 * s;
          is.slab_rt(d0 + TM_LIN, f_img + (uint64_t)(s * (2 * SLAB >> 4)), rem >= 64 ? 4 : (rem + 15) >> 4, acc);
        }
        if (elect_one_sync()) umma_commit(&b->lin_bar);
      }
      // ---- layer 0: the h-parts of r and z do not need x0
      is.gate<true>(d0 + TM_R, h0_img);
      is.gate<true>(d0 + TM_Z, h0_img);
      TWAIT(t_x0, wait_flip(&b->x0_rdy, p_x0));          // x0 image written, D_lin consumed
      tc_fence_after();
      is.gate<true>(d0 + TM_NH, h0_img);
      is.gate<false>(d0 + TM_R, x0_img);
      is.gate<false>(d0 + TM_Z, x0_img);
      is.gate<true>(d0 + TM_NX, x0_img);
      if (elect_one_sync()) umma_commit(&b->d_bar[0]);
      if (L == 2) {
        if (t > 0) { TWAIT(t_h1, wait_flip(&b->h_rdy[1], p_h1)); tc_fence_after(); }   // layer-1 gates of step t-1: D1 free, h1 image new
        is.gate<true>(d1 + TM_R, h1_img);
        is.gate<true>(d1 + TM_Z, h1_img);
        is.gate<true>(d1 + TM_NH, h1_img);
        TWAIT(t_h0, wait_flip(&b->h_rdy[0], p_h0));      // layer-0 gates of this step: new h0 image, D0 free
        tc_fence_after();
        is.gate<false>(d1 + TM_R, h0_img);
        is.gate<false>(d1 + TM_Z, h0_img);
        is.gate<true>(d1 + TM_NX, h0_img);
        if (elect_one_sync()) umma_commit(&b->d_bar[1]);
      } else {
        TWAIT(t_h0, wait_flip(&b->h_rdy[0], p_h0));
        tc_fence_after();
      }
    }
    if (L == 2) { TWAIT(t_h1, wait_flip(&b->h_rdy[1], p_h1)); tc_fence_after(); }    // last step's layer-1 gates
  }
#if GRU_TIMING
  if (blockIdx.x == 0 && (threadIdx.x & 31) == 0)
    printf("issuer: total %lld cycles, waits: weights %lld, features %lld, x0 %lld, h0 %lld, h1 %lld\n", clock64() - t_begin, is.t_w,
           t_f, t_x0, t_h0, t_h1);
#endif
}

// ---------------------------------------------------------------------------------------------- weight ring (one lane)
__device__ __noinline__ void weights_role(const GruTcArgs& a, Bars* b, uint8_t* base, int my_tiles) {
  const int per_step = 2 * ((a.idim + 63) >> 6) + 24 * a.L;
  const long long total = (long long)my_tiles * a.T * per_step;
  int ci = 0;
  uint32_t slot = 0, free_par = 0;
  for (long long c = 0; c < total; ++c) {
    if (c >= NSLOT) {
      mbar_wait(&b->w_free[slot], (free_par >> slot) & 1u);
      free_par ^= 1u << slot;
    }
    mbar_arrive_expect_tx(&b->w_full[slot], CHUNK);
    bulk_g2s(base + OFF_RING + slot * CHUNK, a.wimg + (size_t)ci * CHUNK, CHUNK, &b->w_full[slot]);
    slot = slot + 1 == NSLOT ? 0 : slot + 1;
    ci = ci + 1 == per_step ? 0 : ci + 1;
  }
}

// ------------------------------------------------------------------------------------------------------------- kernel
__global__ void __launch_bounds__(NT, 1) gru_tc_kernel(const __grid_constant__ GruTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  __shared__ Bars bars;
  __shared__ uint32_t tmem_slot;
  const uint32_t sbase = smem_u32(base);
  const int tid = threadIdx.x, warp = __shfl_sync(0xffffffffu, tid >> 5, 0), lane = tid & 31;
  const float* vec = a.vec;
  const int L = a.L, T = a.T;

  if (tid == 0) {
    for (int i = 0; i < NSLOT; ++i) { mbar_init(&bars.w_full[i], 1); mbar_init(&bars.w_free[i], 1); }
    mbar_init(&bars.f_rdy, 2);
    mbar_init(&bars.lin_bar, 1);
    mbar_init(&bars.x0_rdy, 8);
    mbar_init(&bars.d_bar[0], 1); mbar_init(&bars.d_bar[1], 1);
    mbar_init(&bars.h_rdy[0], 8); mbar_init(&bars.h_rdy[1], 8);
    mbar_fence_init();
  }
  if (warp == 8) tmem_alloc(&tmem_slot, TM_COLS);
  // the feature image's K padding must be finite (it meets zero weights): clear it once
  for (int i = tid; i < IMG / 16; i += NT) reinterpret_cast<uint4*>(base + OFF_F)[i] = make_uint4(0, 0, 0, 0);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;

  const int my_tiles = a.n_tiles > (int)blockIdx.x ? (a.n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;

  if (warp == 8) {
    issuer_role(a, &bars, sbase, tmem, my_tiles);
  } else if (warp == 9) {
    if (lane == 0) weights_role(a, &bars, base, my_tiles);
  } else if (warp >= 10) {
    // ---- feature rows: thread = stream row; CMVN (cmvn.py:45-47), bf16 hi|lo split, 16-byte chunks into the image
    const int m = tid - 320;
    uint32_t p_lin = 0;
    long long step = 0;
    for (int it = 0; it < my_tiles; ++it) {
      const int b0 = (blockIdx.x + it * gridDim.x) * a.ms;
      const bool live = m < a.ms && b0 + m < a.B;
      for (int t = 0; t < T; ++t, ++step) {
        float4 f4[24];
        const float* src0 = a.feats + ((size_t)(b0 + m) * T + t) * a.idim;
        const bool vec4 = (a.idim & 3) == 0 && (reinterpret_cast<uintptr_t>(a.feats) & 15) == 0;
#pragma unroll
        for (int i = 0; i < 24; ++i) {
          f4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (live && 4 * i < a.idim) {
            if (vec4) f4[i] = __ldg(reinterpret_cast<const float4*>(src0) + i);
            else {
              f4[i].x = __ldg(src0 + 4 * i);
              if (4 * i + 1 < a.idim) f4[i].y = __ldg(src0 + 4 * i + 1);
              if (4 * i + 2 < a.idim) f4[i].z = __ldg(src0 + 4 * i + 2);
              if (4 * i + 3 < a.idim) f4[i].w = __ldg(src0 + 4 * i + 3);
            }
          }
        }
        if (step > 0) wait_flip(&bars.lin_bar, p_lin);     // the previous step's Linear has read the image
#pragma unroll
        for (int ch = 0; ch < 12; ++ch) {
          if (8 * ch < a.idim) {
            float v[8] = {f4[2 * ch].x, f4[2 * ch].y, f4[2 * ch].z, f4[2 * ch].w,
                          f4[2 * ch + 1].x, f4[2 * ch + 1].y, f4[2 * ch + 1].z, f4[2 * ch + 1].w};
            const int k0 = 8 * ch;
            if (a.has_cmvn && live) {
#pragma unroll
              for (int u = 0; u < 8; ++u)
                if (k0 + u < a.idim) v[u] = (v[u] - __ldg(vec + a.v_mean + k0 + u)) * __ldg(vec + a.v_istd + k0 + u);
            }
            const uint32_t off = a_off(m, k0);
            split_store8(v, base + OFF_F, base + OFF_F + SLAB, off);
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.f_rdy);
      }
    }
  } else {
    // ---- unit owners: thread = (hidden unit j, 32 streams)
    const int q = warp & 3, sh = warp >> 2;
    const int j = 32 * q + lane;
    const uint32_t trow = tmem + ((uint32_t)(32 * q) << 16);
    const int s0 = 32 * sh;                                  // first stream of this thread
    // image address pieces of K element j: row m adds m * 128 and flips the 16-byte chunk by (m & 7)
    const uint32_t kbase = (uint32_t)((j >> 6) * 2 * SLAB + (j & 7) * 2);
    const uint32_t kc16 = (uint32_t)(((j & 63) >> 3) << 4);
    uint32_t p_lin = 0, p_d0 = 0, p_d1 = 0, p_h = 0;
    float hreg[2][32];
    long long t_lin = 0, t_d0 = 0, t_d1 = 0, t_cls = 0, s_pro = 0, s_x0 = 0, s_g0 = 0, s_g1 = 0, s_cls = 0, s_fin = 0;
    const long long t_begin = clock64();
    for (int it = 0; it < my_tiles; ++it) {
      const int b0 = (blockIdx.x + it * gridDim.x) * a.ms;
      const int Mv = min(a.ms, a.B - b0);                    // live streams of the tile (rows Mv.. of the images are never read back)
      const int nchunk = Mv <= s0 ? 0 : Mv - s0 <= 16 ? 1 : 2;   // 16-stream chunks of this thread that hold live streams
      // ---- initial hidden state -> fp32 registers + operand images
      TSEG_BEGIN(tp0)
#pragma unroll
      for (int l = 0; l < 2; ++l) {                          // compile-time l: hreg stays in registers
        if (l >= L) break;
        {
          const float* hin = a.in_cache != nullptr ? a.in_cache + ((size_t)l * a.B + b0 + s0) * H + j : nullptr;
          const int nlive = hin != nullptr ? Mv - s0 : 0;    // streams of this thread that exist
#pragma unroll
          for (int i = 0; i < 32; ++i) hreg[l][i] = i < nlive ? __ldg(hin + i * H) : 0.f;
        }
        uint8_t* img = base + OFF_H + l * IMG + kbase;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          if (c >= nchunk) break;
#pragma unroll
          for (int i = 16 * c; i < 16 * c + 16; ++i) {
            uint16_t hi, lo;
            split1(hreg[l][i], hi, lo);
            const uint32_t off = (uint32_t)((s0 + i) * 128) + (kc16 ^ (uint32_t)((i & 7) << 4));
            *reinterpret_cast<uint16_t*>(img + off) = hi;
            *reinterpret_cast<uint16_t*>(img + off + SLAB) = lo;
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.h_rdy[l]);
      }
      TSEG_END(s_pro, tp0)
      wait_flip(&bars.h_rdy[L - 1], p_h);                    // (keeps this thread's phase count of the barrier in step)
      const float bp = __ldg(vec + a.v_bp + j);
      for (int t = 0; t < T; ++t) {
        // ================= x0 = relu(Linear + b)  -> X0 image
        TWAIT(t_lin, wait_flip(&bars.lin_bar, p_lin));
        tc_fence_after();
        TSEG_BEGIN(tx0)
        {
          uint8_t* img = base + OFF_X0 + kbase;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (c >= nchunk) break;
            float d[16];
            tmem_ld16(trow + TM_LIN + s0 + 16 * c, d);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              uint16_t hi, lo;
              split1(fmaxf(d[i] + bp, 0.f), hi, lo);
              const uint32_t off = (uint32_t)((s0 + 16 * c + i) * 128) + (kc16 ^ (uint32_t)((i & 7) << 4));
              *reinterpret_cast<uint16_t*>(img + off) = hi;
              *reinterpret_cast<uint16_t*>(img + off + SLAB) = lo;
            }
          }
        }
        tc_fence_before();
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars.x0_rdy);
        TSEG_END(s_x0, tx0)
        // ================= GRU layers
#pragma unroll
        for (int l = 0; l < 2; ++l) {
          if (l >= L) break;
          const float* bih = vec + a.v_layers + (size_t)l * a.v_layer_stride + 2 * H * 3 * H;   // b_ih (384) then b_hh (384)
          const float* bhh = bih + 3 * H;
          const float nb_r = -LOG2E * (__ldg(bih + j) + __ldg(bhh + j)), nb_z = -LOG2E * (__ldg(bih + H + j) + __ldg(bhh + H + j));
          const float b_nx = __ldg(bih + 2 * H + j), b_nh = __ldg(bhh + 2 * H + j);
          if (l == 0) { TWAIT(t_d0, wait_flip(&bars.d_bar[0], p_d0)); } else { TWAIT(t_d1, wait_flip(&bars.d_bar[1], p_d1)); }
          tc_fence_after();
          TSEG_BEGIN(tg)
          const uint32_t td = trow + TM_LAYER * l + s0;
          uint8_t* img = base + OFF_H + l * IMG + kbase;
#pragma unroll
          for (int c = 0; c < 2; ++c) {
            if (c >= nchunk) break;
            float gr[16], gz[16], gx[16], gh[16];
            tmem_ld16(td + TM_R + 16 * c, gr);
            tmem_ld16(td + TM_Z + 16 * c, gz);
            tmem_ld16(td + TM_NX + 16 * c, gx);
            tmem_ld16(td + TM_NH + 16 * c, gh);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float r = sigmoid_fast(gr[i], nb_r);
              const float z = sigmoid_fast(gz[i], nb_z);
              const float n = tanh_fast(fmaf(r, gh[i] + b_nh, gx[i] + b_nx));
              const float hn = n + z * (hreg[l][16 * c + i] - n);   // (1 - z) n + z h
              hreg[l][16 * c + i] = hn;
              uint16_t hi, lo;
              split1(hn, hi, lo);
              const uint32_t off = (uint32_t)((s0 + 16 * c + i) * 128) + (kc16 ^ (uint32_t)((i & 7) << 4));
              *reinterpret_cast<uint16_t*>(img + off) = hi;
              *reinterpret_cast<uint16_t*>(img + off + SLAB) = lo;
            }
          }
          tc_fence_before();
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&bars.h_rdy[l]);
          if (l == 0) { TSEG_END(s_g0, tg) } else { TSEG_END(s_g1, tg) }
        }
        // ================= classifier on the top layer's h_t (classifier.py:54-67): one warp per (stream, output)
        TWAIT(t_cls, wait_flip(&bars.h_rdy[L - 1], p_h));    // every unit of the new top h is in the image
        TSEG_BEGIN(tc0)
        {
          // 8 (stream, output) pairs per warp pass: lanes split k, the 8 reductions run interleaved, then lane i finishes
          // pair i (bias, activation, store) -- one latency chain per pass instead of one per pair
          const uint8_t* img = base + OFF_H + (L - 1) * IMG;
          const int npair = Mv * a.odim;
          for (int o0 = 8 * warp; o0 < npair; o0 += 64) {
            float acc[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int o = min(o0 + i, npair - 1);
              const int ms = a.odim == 1 ? o : o / a.odim, jo = a.odim == 1 ? 0 : o - ms * a.odim;
              const float* wc = vec + a.v_wc + jo;             // WcT[k][odim]
              float v = 0.f;
#pragma unroll
              for (int u = 0; u < H / 32; ++u) {
                const int k = lane + 32 * u;
                const uint32_t off = a_off(ms, k);
                const float hv = __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(img + off)) +
                                 __bfloat162float(*reinterpret_cast<const __nv_bfloat16*>(img + off + SLAB));
                v = fmaf(__ldg(wc + k * a.odim), hv, v);
              }
              acc[i] = v;
            }
#pragma unroll
            for (int sft = 16; sft > 0; sft >>= 1)
#pragma unroll
              for (int i = 0; i < 8; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], sft);
            float mine = acc[0];
#pragma unroll
            for (int i = 1; i < 8; ++i) mine = lane == i ? acc[i] : mine;
            const int o = o0 + lane;
            if (lane < 8 && o < npair) {
              const int ms = a.odim == 1 ? o : o / a.odim, jo = a.odim == 1 ? 0 : o - ms * a.odim;
              mine += __ldg(vec + a.v_bc + jo);
              if (a.act == WEKWS_ACT_SIGMOID) mine = sigmoidf_acc(mine);
              a.out[((size_t)(b0 + ms) * T + t) * a.odim + jo] = mine;
            }
          }
        }
        TSEG_END(s_cls, tc0)
      }
      // ---- final hidden state
      TSEG_BEGIN(tf0)
#pragma unroll
      for (int l = 0; l < 2; ++l) {
        if (l >= L) break;
        float* hout = a.out_cache + ((size_t)l * a.B + b0 + s0) * H + j;
        const int nlive = Mv - s0;
#pragma unroll
        for (int i = 0; i < 32; ++i)
          if (i < nlive) hout[i * H] = hreg[l][i];
      }
      // the top layer's image is rewritten by the next tile's prologue: every owner must be done with its classifier
      // reads (named barrier among the 256 owners)
      TSEG_END(s_fin, tf0)
      asm volatile("bar.sync 1, 256;" ::: "memory");
    }
#if GRU_TIMING
    if (blockIdx.x == 0 && tid == 0)
      printf("owner: total %lld cycles, waits: lin %lld, d0 %lld, d1 %lld, top-h %lld; busy: prologue %lld, x0 %lld, gates0 %lld, gates1 %lld, classifier %lld, final %lld\n",
             clock64() - t_begin, t_lin, t_d0, t_d1, t_cls, s_pro, s_x0, s_g0, s_g1, s_cls, s_fin);
#endif
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

size_t gru_tc_image_bytes(int L, int idim) { return (size_t)(2 * ((idim + 63) / 64) + 24 * L) * CHUNK; }

bool gru_tc_eligible(int L, int H_, int idim) { return H_ == H && (L == 1 || L == 2) && idim >= 1 && idim <= 96; }

// host: the per-step weight stream, in the order the MMA issuer consumes it.  Every chunk is a K-major SWIZZLE_128B
// bf16 image of 128 rows (hidden units) x 64 K (tc_common.cuh layout: row n at n*128, 16-byte chunk c of the slab at
// chunk c ^ (n & 7)); per K slab a hi chunk then a lo chunk.  Order: Linear; per layer W_hh (r, z, n) then W_ih (r, z, n).
void gru_tc_pack(uint8_t* dst, const float* wp /*[H][idim]*/, int idim, const float* const* wih /*[L] of [3H][H]*/,
                 const float* const* whh, int L) {
  uint8_t* p = dst;
  auto slab = [&](const float* W, int ld, int row0, int k0, int kn) {    // rows row0..row0+127, K k0..k0+kn-1
    write_sw128_image(p, CHUNK, W + (size_t)row0 * ld + k0, H, (size_t)ld, 1, kn);
    p += 2 * CHUNK;
  };
  for (int s = 0; s * 64 < idim; ++s) slab(wp, idim, 0, 64 * s, idim - 64 * s < 64 ? idim - 64 * s : 64);
  for (int l = 0; l < L; ++l) {
    for (int g = 0; g < 3; ++g)
      for (int s = 0; s < 2; ++s) slab(whh[l], H, g * H, 64 * s, 64);
    for (int g = 0; g < 3; ++g)
      for (int s = 0; s < 2; ++s) slab(wih[l], H, g * H, 64 * s, 64);
  }
}

int gru_tc_launch(GruTcArgs a, cudaStream_t st) {
  WEKWS_REQUIRE(a.B >= 1 && a.T >= 1, "gru_tc_launch: empty call");
  // streams per tile: fewer streams per CTA shorten the gate math on the critical path of a step (it is SFU-bound: six
  // ex2 / rcp per unit and stream), the weight stream per CTA and step is the same 786 KB whatever the tile holds
  const int sms0 = device_sm_count();
  a.ms = a.B > 32 * sms0 ? 64 : a.B > 16 * sms0 ? 32 : 16;
  if (const char* e = getenv("WEKWS_GRU_MS")) { const int v = atoi(e); if (v == 16 || v == 32 || v == 64) a.ms = v; }
  a.n_tiles = (a.B + a.ms - 1) / a.ms;
  static bool attr_set[64] = {false};
  if (int rc = set_max_dynamic_smem_once(attr_set, SMEM_BYTES, gru_tc_kernel)) return rc;
  const int sms = device_sm_count();
  const int grid = a.n_tiles < sms ? a.n_tiles : sms;
  gru_tc_kernel<<<grid, NT, SMEM_BYTES, st>>>(a);
  return check_launch("gru_tc_kernel");
}

}  // namespace wekws
