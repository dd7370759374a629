// Tensor-core (tcgen05 / TMEM) fused forward for the depthwise-separable TCN backbone with hidden_dim 256
// (reference wekws/model/tcn.py:91-119 DsCnnBlock inside TCN :122-166, ds_tcn.yaml; BatchNorm folded):
//     per block:  a = ReLU(dw_k8,dil(cat(cache, x)))   o = ReLU(W_pw . a + b)   x' = o + x
// The pointwise 256x256 GEMM carries 97 % of the FLOPs and runs on tcgen05 with the bf16x3 split; the
// depthwise taps, BN/ReLU/residual and the classifier stay in FP32 on the CUDA cores.
//
// One CTA per SM owns a tile of up to 120 frames (spt = 120 / T whole streams) for the whole network:
//   * X[256][120] fp32, the residual stream (frames only), lives in shared memory (120 KB);
//   * the cache (halo) columns of a block are NOT staged: 256 channels x 56 columns x 3 streams would not fit
//     next to X, so the depthwise taps that reach back before the chunk read the cache straight from
//     global memory (lanes = consecutive frames, so a warp reads contiguous floats of one cache row);
//   * the depthwise output is produced 64 channels (one K slab) at a time, split into bf16 hi/lo and written
//     to one of two TMEM operand buffers (tcgen05.st), so slab ks+1 is computed while the MMAs of slab ks run;
//   * the accumulator D[128][256] fp32 lives in TMEM (256 columns); every slab issues, for each half of the
//     output channels, 3 x 4 MMAs (M=128, N=128, K=16) whose B operand is a pre-swizzled 32 KB weight image
//     streamed from L2 through a 3-slot ring by cp.async.bulk (the 256 KB of a block's weights do not fit);
//   * depthwise coefficients of the current block (9 KB) are staged by one bulk copy per block.
// Warp roles: 16 compute warps (row = 32 * (warp % 4) + lane, channel group = warp / 4) + 1 issuer warp.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "dstcn_tc.h"
#include "tc_common.cuh"

namespace wekws {

namespace {

using namespace tc;

constexpr int NCW = 16, NCT = NCW * 32, NT_TC = NCT + 32;
constexpr int C = 256, KT = 8;
constexpr int RPX = 120;                                   // frames per tile == row pitch of X
constexpr int X_BYTES = C * RPX * 4;                       // 122880
constexpr int W_SLOT = 32768, NW = 3;
constexpr int COEF_FLOATS = (KT + 1) * C;                  // [tap][channel] then folded bias
constexpr int OFF_W = 0, OFF_X = NW * W_SLOT, OFF_COEF = OFF_X + X_BYTES;
constexpr int SMEM_TOTAL = OFF_COEF + COEF_FLOATS * 4 + 1024;   // 231424
// TMEM columns: [0,256) accumulator; operand buffer b: hi at 256 + 64 b, lo at 288 + 64 b;
// the first Linear (K <= 128) uses hi at 256.., lo at 320..
constexpr int TM_A = 256, TM_COLS = 512;

__device__ __forceinline__ void compute_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory"); }
__device__ __forceinline__ float ld_global_f32(const float* p) {
  float v;
  asm("ld.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
// predicated global load: 0 when pred == 0 (the address is then not dereferenced)
__device__ __forceinline__ float ld_global_f32_pred(const float* p, uint32_t pred) {
  float v;
  asm volatile(
      "{\n\t"
      ".reg .pred q;\n\t"
      "setp.ne.b32 q, %2, 0;\n\t"
      "mov.f32 %0, 0f00000000;\n\t"
      "@q ld.global.f32 %0, [%1];\n\t"
      "}"
      : "=f"(v)
      : "l"(p), "r"(pred));
  return v;
}
__device__ __forceinline__ void split_to_tmem(const float (&v)[8], uint32_t t_hi, uint32_t t_lo) {
  uint32_t h[4], l[4];
  split2(v[0], v[1], h[0], l[0]); split2(v[2], v[3], h[1], l[1]);
  split2(v[4], v[5], h[2], l[2]); split2(v[6], v[7], h[3], l[3]);
  tmem_st4(t_hi, h);
  tmem_st4(t_lo, l);
}

// PP: compile-time cache row pitch (floats) so the cache loads get immediate offsets; 0 = read it from the arguments
template <int PP>
__global__ void __launch_bounds__(NT_TC, 1) dstcn_tc_kernel(const DsTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  __shared__ uint64_t mma_bar, coef_bar, a_rdy[2], ab_free[2], w_bar[NW], w_free[NW];
  __shared__ uint32_t tmem_slot;
  __shared__ int store_ctr[1];

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer = warp == NCW;
  const int q = warp & 3, g = (warp >> 2) & 3;
  const int row = 32 * q + lane;
  const int T = a.T, P = PP ? PP : a.P;
  const float* vec = a.vec;
  float* X = reinterpret_cast<float*>(base + OFF_X);
  float* coef = reinterpret_cast<float*>(base + OFF_COEF);
  uint8_t* Wring = base + OFF_W;

  if (tid == 0) {
    mbar_init(&mma_bar, 1); mbar_init(&coef_bar, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&a_rdy[i], NCW); mbar_init(&ab_free[i], 1); }
    for (int i = 0; i < NW; ++i) { mbar_init(&w_bar[i], 1); mbar_init(&w_free[i], 1); }
    mbar_fence_init();
  }
#ifdef WEKWS_MBAR_WATCHDOG
  if (tid == 0 && blockIdx.x == 0)
    printf("dstcn_tc barriers: mma_bar 0x%x coef_bar 0x%x a_rdy 0x%x ab_free 0x%x w_bar 0x%x w_free 0x%x\n", smem_u32(&mma_bar),
           smem_u32(&coef_bar), smem_u32(a_rdy), smem_u32(ab_free), smem_u32(w_bar), smem_u32(w_free));
#endif
  if (is_issuer) tmem_alloc(&tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform32(tmem_slot);      // warp-uniform: MMA operands are then built in uniform registers
  uint32_t mma_par = 0, coef_par = 0;
  const uint32_t idesc = make_idesc_bf16(128, 128);
  const int natoms = (a.idim + 63) / 64;
  const int spt = a.spt;
  const int nlin = 2 * natoms;
  const int nitems = nlin + a.nblocks * 8;          // weight images per pass

  const int sb = (int)(((long long)a.B * blockIdx.x) / gridDim.x);
  const int se = (int)(((long long)a.B * (blockIdx.x + 1)) / gridDim.x);
  const int npass = (se - sb + spt - 1) / spt;
  int done = sb;

  // issuer state: weight items form one continuous sequence over all passes of this CTA (item % nitems = image)
  uint32_t gl = 0, gu = 0, ar_par = 0;
  const uint32_t gtotal = (uint32_t)npass * (uint32_t)nitems;
  auto load_next = [&]() {
    if (gl >= gtotal) return;
    const uint32_t slot = gl % NW, n = gl % (uint32_t)nitems;
    if (lane == 0) {
      mbar_arrive_expect_tx(&w_bar[slot], W_SLOT);
      bulk_g2s(Wring + slot * W_SLOT, a.wimg + (size_t)n * W_SLOT, W_SLOT, &w_bar[slot]);
    }
    ++gl;
  };
  // the cache of the streams of a pass is pulled into L2 one pass ahead, so the depthwise taps that read it
  // straight from global memory see L2 latency instead of HBM latency
  auto prefetch_cache = [&](int first, int n) {
    if (!a.prefetch_ok || lane != 0) return;
    for (int i = 0; i < n; ++i)
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(a.in_cache + (size_t)(first + i) * C * P),
                   "r"(C * P * 4)
                   : "memory");
  };
  if (is_issuer) {                                   // whole warp: uniform bookkeeping, lane 0 issues the copies
    for (int i = 0; i < NW; ++i) load_next();
    prefetch_cache(sb, min(spt, se - sb));
  }

  while (done < se) {
    const int remaining = se - done;
    const int passes_left = (remaining + spt - 1) / spt;
    const int ns = (remaining + passes_left - 1) / passes_left;
    const int b0 = done;
    done += ns;
    const int rows = ns * T;

    if (is_issuer) {
      // ================================================================== MMA-ISSUE WARP
      // All lanes run the (uniform) control flow and descriptor arithmetic; the tcgen05 / bulk-copy instructions are
      // elected.  With `if (lane == 0)` around the whole role every MMA sat in an ELECT / R2UR waterfall loop.
      {
        // D[:, d_col .. d_col+128) (+)= A(tmem a_hi / a_lo, ksteps K-steps) x W(next image)   -- bf16x3
        auto use_item = [&](uint32_t d_col, uint32_t a_hi, uint32_t a_lo, int ksteps, uint32_t& acc) {
          const uint32_t slot = gu % NW;
          mbar_wait(&w_bar[slot], (gu / NW) & 1);
          const uint64_t dwh = make_sdesc_sw128(smem_u32(Wring + slot * W_SLOT)), dwl = dwh + (16384 >> 4);
          const uint32_t d = tmem + d_col, ahi = tmem + a_hi, alo = tmem + a_lo;
          if (elect_one_sync()) {
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, ahi + 8 * k, dwh + 2 * k, idesc, k == 0 ? acc : 1u);
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, alo + 8 * k, dwh + 2 * k, idesc, 1);
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, ahi + 8 * k, dwl + 2 * k, idesc, 1);
            umma_commit(&w_free[slot]);
          }
          acc = 1;
          if (gu >= 1) {                              // the previous image's MMAs are (nearly) done: refill its slot
            mbar_wait(&w_free[(gu - 1) % NW], ((gu - 1) / NW) & 1);
            load_next();
          }
          ++gu;
        };
        auto wait_a = [&](int b) {
          mbar_wait(&a_rdy[b], (ar_par >> b) & 1);
          ar_par ^= 1u << b;
          tc_fence_after();
        };
        auto load_coef = [&](int blk) {
          if (lane == 0) {
            fence_proxy_async();                      // the area was read/written through the generic proxy
            mbar_arrive_expect_tx(&coef_bar, COEF_FLOATS * 4);
            bulk_g2s(coef, vec + a.v_blocks + (size_t)blk * a.v_blk_stride, COEF_FLOATS * 4, &coef_bar);
          }
        };
        load_coef(0);
        if (done < se) prefetch_cache(done, min(spt, se - done));
        // ---- first Linear
        {
          const int ks0 = (min(a.idim, 64) + 15) >> 4, ks1 = natoms > 1 ? (a.idim - 64 + 15) >> 4 : 0;
          wd_mark(100);
          wait_a(0);
          uint32_t acc0 = 0, acc1 = 0;
          use_item(0, TM_A, TM_A + 64, ks0, acc0);
          use_item(128, TM_A, TM_A + 64, ks0, acc1);
          if (natoms > 1) {
            use_item(0, TM_A + 32, TM_A + 96, ks1, acc0);
            use_item(128, TM_A + 32, TM_A + 96, ks1, acc1);
          }
          if (elect_one_sync()) umma_commit(&mma_bar);
        }
        // ---- blocks: K slab ks of block blk
        for (int blk = 0; blk < a.nblocks; ++blk) {
          for (int ks = 0; ks < 4; ++ks) {
            const int b = ks & 1;
            wd_mark(1000 + blk * 10 + ks);
            wait_a(b);
            wd_mark(2000 + blk * 10 + ks);
            if (ks == 3 && blk + 1 < a.nblocks) load_coef(blk + 1);   // every warp is past this block's taps
            uint32_t acc0 = ks > 0 ? 1u : 0u, acc1 = acc0;
            use_item(0, TM_A + 64 * b, TM_A + 32 + 64 * b, 4, acc0);
            use_item(128, TM_A + 64 * b, TM_A + 32 + 64 * b, 4, acc1);
            if (elect_one_sync()) {
              umma_commit(&ab_free[b]);
              if (ks == 3) umma_commit(&mma_bar);
            }
          }
        }
        wd_mark(3000);
      }
    } else {
      // ================================================================== COMPUTE WARPS
      // Rows are ordered frame-major: row = t * ns + s, and X[c][row] likewise, so a tap is a column shift of
      // j * d * ns and the rows of a warp span ~32 / ns consecutive frames: only the warps holding the first frames
      // of the chunk reach back into the cache, and only for their first taps.
      const bool valid = row < rows, q_live = 32 * q < rows;
      const int t = valid ? row / ns : 0, s = valid ? row - t * ns : 0;
      const int t_min = (32 * q) / ns;                 // first frame of this warp's rows
      const uint32_t tm_row = tmem + ((uint32_t)(32 * q) << 16);

      auto hand_over = [&](int b) {
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_rdy[b]);
      };
      auto wait_mma = [&]() {
        mbar_wait(&mma_bar, mma_par);
        mma_par ^= 1u;
        tc_fence_after();
      };

      // ---- features (+CMVN) -> bf16 hi/lo operand of the first Linear
      wd_mark(1);
      if (q_live) {
        const int nch = ((a.idim + 15) >> 4) * 2;
        const float* src0 = a.feats + (size_t)(b0 + s) * a.feat_bstride + (size_t)t * a.idim;
        for (int ch = g; ch < nch; ch += 4) {
          float v[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) v[u] = 0.f;
          const int k0 = ch * 8;
          if (valid && k0 < a.idim) {
            const float4 f0 = __ldg(reinterpret_cast<const float4*>(src0 + k0));
            const float4 f1 = __ldg(reinterpret_cast<const float4*>(src0 + k0) + 1);
            v[0] = f0.x; v[1] = f0.y; v[2] = f0.z; v[3] = f0.w; v[4] = f1.x; v[5] = f1.y; v[6] = f1.z; v[7] = f1.w;
            if (a.has_cmvn) {
#pragma unroll
              for (int u = 0; u < 8; ++u) v[u] = (v[u] - __ldg(vec + a.v_mean + k0 + u)) * __ldg(vec + a.v_istd + k0 + u);
            }
          }
          split_to_tmem(v, tm_row + TM_A + 4 * ch, tm_row + TM_A + 64 + 4 * ch);
        }
      }
      hand_over(0);
      wd_mark(2);
      // ---- x = relu(D + bp) -> X
      wait_mma();
      if (q_live) {
#pragma unroll 1
        for (int i4 = 0; i4 < 4; ++i4) {
          const int c0 = 64 * g + 16 * i4;
          float d[16];
          tmem_ld16(tm_row + c0, d);
          if (valid) {
            const float4* bp4 = reinterpret_cast<const float4*>(vec + a.v_bp + c0);
#pragma unroll
            for (int e4 = 0; e4 < 4; ++e4) {
              const float4 bv = __ldg(bp4 + e4);
              const float bb[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
              for (int u = 0; u < 4; ++u) X[(c0 + 4 * e4 + u) * RPX + row] = fmaxf(d[4 * e4 + u] + bb[u], 0.f);
            }
          }
        }
      }
      if (tid == 0) store_ctr[0] = 0;
      tc_fence_before();
      compute_barrier();
      wd_mark(3);

      for (int blk = 0; blk < a.nblocks; ++blk) {
        const int d = a.dil[blk], pad = d * (KT - 1), off = a.coff[blk];
        mbar_wait(&coef_bar, coef_par);
        coef_par ^= 1u;
        // taps that reach back before the chunk read cat index < pad from the cache row of this stream
        const float* crow = valid && a.in_cache != nullptr ? a.in_cache + (size_t)(b0 + s) * C * P + off : nullptr;
        const int t0 = valid ? t : -(1 << 20);         // padding rows: every cache-capable tap takes the absent-cache path
        // taps j < jc can need the cache for some row of this warp (t_min + j d < pad); rounded up to a compiled variant
        const int jc = pad > t_min ? min(KT - 1, (pad - t_min + d - 1) / d) : 0;

        // depthwise taps of 8 channels -> ReLU -> bf16 hi/lo -> TMEM operand buffer b.  Taps j < JC are compiled with
        // a predicated global load (cache part) next to the shared load (frame part), the rest with the shared load
        // only; everything is branch-free so the loads of a chunk are in flight together.
        auto dw_chunk = [&](auto jct, int c0, uint32_t t_hi, uint32_t t_lo) {
          constexpr int JC = decltype(jct)::value;
          float acc[8];
          {
            const float4 b0v = *reinterpret_cast<const float4*>(coef + KT * C + c0);
            const float4 b1v = *reinterpret_cast<const float4*>(coef + KT * C + c0 + 4);
            acc[0] = b0v.x; acc[1] = b0v.y; acc[2] = b0v.z; acc[3] = b0v.w;
            acc[4] = b1v.x; acc[5] = b1v.y; acc[6] = b1v.z; acc[7] = b1v.w;
          }
          const float* xc = X + c0 * RPX + row;
          const float* gc = crow + (size_t)c0 * P + t0;
#pragma unroll
          for (int j = 0; j < KT; ++j) {
            const float4 w0 = *reinterpret_cast<const float4*>(coef + j * C + c0);
            const float4 w1 = *reinterpret_cast<const float4*>(coef + j * C + c0 + 4);
            const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
            const int sh = (j * d - pad) * ns;         // column shift of the frame part
            float v[8];
            if (j < JC) {
              const bool in_c = t0 + j * d < pad, pg = in_c && crow != nullptr;
              const float* xp = in_c ? X + c0 * RPX : xc + sh;
              const float* gp = gc + j * d;
#pragma unroll
              for (int u = 0; u < 8; ++u) {
                const float vx = xp[u * RPX];
                const float vg = pg ? ld_global_f32(gp + u * P) : 0.f;   // L1-cached: neighbouring taps/rows re-read it
                v[u] = in_c ? vg : vx;
              }
            } else {
#pragma unroll
              for (int u = 0; u < 8; ++u) v[u] = xc[sh + u * RPX];
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) acc[u] = fmaf(w[u], v[u], acc[u]);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) acc[u] = fmaxf(acc[u], 0.f);
          split_to_tmem(acc, t_hi, t_lo);
        };

        for (int ks = 0; ks < 4; ++ks) {
          const int b = ks & 1;
          wd_mark(10000 + blk * 10 + ks);
          if (ks >= 2) {                               // the MMAs of slab ks-2 have drained this operand buffer
            mbar_wait(&ab_free[b], 0);                 // (two commits per buffer and block: always the even phase)
            tc_fence_after();
          }
          wd_mark(20000 + blk * 10 + ks);
          if (q_live) {
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
              const int c0 = 64 * ks + 16 * g + 8 * half;
              const uint32_t t_hi = tm_row + TM_A + 64 * b + 4 * (2 * g + half), t_lo = t_hi + 32;
              if (jc == 0) dw_chunk(std::integral_constant<int, 0>{}, c0, t_hi, t_lo);
              else if (jc <= 3) dw_chunk(std::integral_constant<int, 3>{}, c0, t_hi, t_lo);
              else if (jc <= 5) dw_chunk(std::integral_constant<int, 5>{}, c0, t_hi, t_lo);
              else dw_chunk(std::integral_constant<int, 7>{}, c0, t_hi, t_lo);
            }
          }
          if (ks == 3) {
            // New cache slices (tcn.py:54: last `pad` columns of cat(cache, x)), stored before this warp's last
            // hand-over so the epilogue (which overwrites x) cannot start before every store has been issued.  x is
            // stable during the whole depthwise phase, so a warp starts as soon as its own taps are done and takes
            // row groups from a shared counter: the warps without cache taps finish early and do most of the moving.
            // Only when out_cache aliases in_cache must every warp first be past its last read of the old slices.
            if (a.aliased) compute_barrier();
            const int L = pad <= 8 ? 8 : pad <= 16 ? 16 : 32, npr = 32 / L, sub = lane / L, pl = lane - sub * L;
            const int ngroups = ns * C / npr;          // a group = npr rows of `pad` floats, one warp iteration per L floats
            const size_t pbase = (size_t)b0 * C * P + off;
            const float* ic = a.in_cache != nullptr ? a.in_cache + pbase : nullptr;
            float* oc = a.out_cache + pbase;
            const int from_cache = pad - T;            // elements p < pad - T come from the old slice (column p + T)
            for (;;) {
              int g0 = 0;
              if (lane == 0) g0 = atomicAdd(store_ctr, 4);
              g0 = __shfl_sync(0xffffffffu, g0, 0);
              if (g0 >= ngroups) break;
              const int g1 = min(g0 + 4, ngroups);
              for (int gi = g0; gi < g1; ++gi) {
                const int r = gi * npr + sub, ss = r >> 8, c = r & (C - 1), rp = r * P;
                const float* xrow = X + c * RPX + ss + (T - pad) * ns;      // element p of the new slice = xrow[p * ns]
                for (int p0 = 0; p0 < pad; p0 += L) {  // ascending: a row shifts left by T, reads stay ahead of writes
                  const int p = p0 + pl;
                  const bool act = p < pad, fx = p >= from_cache;
                  const float xv = xrow[(act && fx ? p : pad - T) * ns];
                  float v = 0.f;
                  if (act && !fx && ic != nullptr) v = __ldcg(ic + rp + T + p);
                  v = fx ? xv : v;
                  if (a.aliased) __syncwarp();
                  if (act) oc[rp + p] = v;
                }
              }
            }
          }
          hand_over(b);
        }
        // ---- x' = relu(D + b_pw) + x -> X                                   (tcn.py:60: no ReLU after the add)
        wd_mark(30000 + blk);
        wait_mma();
        if (q_live) {
          const float* bb = vec + a.v_blocks + blk * a.v_blk_stride + (KT + 1) * C;
#pragma unroll 1
          for (int i4 = 0; i4 < 4; ++i4) {
            const int c0 = 64 * g + 16 * i4;
            float dd[16];
            tmem_ld16(tm_row + c0, dd);
            if (valid) {
              const float4* b4 = reinterpret_cast<const float4*>(bb + c0);
#pragma unroll
              for (int e4 = 0; e4 < 4; ++e4) {
                const float4 bv = __ldg(b4 + e4);
                const float bq[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  float* xp = X + (c0 + 4 * e4 + u) * RPX + row;
                  *xp = fmaxf(dd[4 * e4 + u] + bq[u], 0.f) + *xp;
                }
              }
            }
          }
        }
        if (tid == 0) store_ctr[0] = 0;
        tc_fence_before();
        compute_barrier();
      }

      // ---- classifier + activation on x (tcn.py:165 -> classifier.py:63-67); partial sums reuse the coefficient area
      wd_mark(40000);
      const int odim = a.odim;
      if (a.hidden != nullptr) {
        // wide classifier heads run as their own tcgen05 GEMM (linear_tc.cu): hand over x as (stream, frame, 256) rows.
        // lanes = consecutive rows (conflict-free reads of X[c][row]); each warp walks the channels
        for (int c = warp; c < C; c += NCW) {
          for (int r = lane; r < rows; r += 32) {
            const int tt = r / ns, ss = r - tt * ns;
            a.hidden[(size_t)(b0 + ss) * a.hidden_bstride + (size_t)tt * C + c] = X[c * RPX + r];
          }
        }
      } else {
      {
        const int r = tid & 127, part = tid >> 7;
        if (r < rows) {
          for (int j = 0; j < odim; ++j) {
            float y = 0.f;
#pragma unroll 8
            for (int c = 64 * part; c < 64 * part + 64; ++c) y = fmaf(__ldg(vec + a.v_wc + c * odim + j), X[c * RPX + r], y);
            coef[(j * 4 + part) * 128 + r] = y;
          }
        }
      }
      compute_barrier();
      for (int idx = tid; idx < rows * odim; idx += NCT) {
        const int r = idx / odim, j = idx - r * odim;
        float y = __ldg(vec + a.v_bc + j) + coef[(j * 4 + 0) * 128 + r] + coef[(j * 4 + 1) * 128 + r] +
                  coef[(j * 4 + 2) * 128 + r] + coef[(j * 4 + 3) * 128 + r];
        if (a.act == WEKWS_ACT_SIGMOID) y = sigmoidf_acc(y);
        const int tt = r / ns, ss = r - tt * ns;
        a.out[(size_t)(b0 + ss) * a.out_bstride + (size_t)tt * odim + j] = y;
      }
    }
      }
    __syncthreads();       // pass boundary
  }

  tc_fence_before();
  __syncthreads();
  if (is_issuer) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

bool dstcn_tc_eligible(const DsTcArgs& a, int hdim) {
  return hdim == C && a.ktaps == KT && a.idim % 8 == 0 && a.idim >= 8 && a.idim <= 128 && a.odim >= 1 && (a.odim <= 4 || a.hidden != nullptr) &&
         a.v_blocks % 4 == 0 && a.v_blk_stride % 4 == 0;
}

int dstcn_tc_max_T() { return RPX; }

int dstcn_tc_launch(DsTcArgs a, cudaStream_t st) {
  WEKWS_REQUIRE(a.T >= 1 && a.T <= RPX && a.B >= 1, "dstcn_tc_launch: bad shape");
  a.spt = RPX / a.T;
  a.prefetch_ok = a.in_cache != nullptr && ((uintptr_t)a.in_cache & 15) == 0 && (C * a.P * 4) % 16 == 0 &&
                  getenv("WEKWS_DS_PREFETCH") != nullptr;      // measured: no gain on B200 (0.357 vs 0.351 ms), off by default
  {
    const size_t bytes = (size_t)a.B * C * a.P * sizeof(float);
    const char* i0 = reinterpret_cast<const char*>(a.in_cache);
    const char* o0 = reinterpret_cast<const char*>(a.out_cache);
    a.aliased = a.in_cache != nullptr && i0 < o0 + bytes && o0 < i0 + bytes;
  }
  const int sms = device_sm_count();
  const int tiles = (a.B + a.spt - 1) / a.spt;
  const int grid = tiles < sms ? tiles : sms;
  static bool attr_set[64] = {false};
  if (int rc = set_max_dynamic_smem_once(attr_set, SMEM_TOTAL, dstcn_tc_kernel<105>, dstcn_tc_kernel<0>)) return rc;
  if (a.P == 105) dstcn_tc_kernel<105><<<grid, NT_TC, SMEM_TOTAL, st>>>(a);     // ds_tcn.yaml: k = 8, dilations 1, 2, 4, 8
  else dstcn_tc_kernel<0><<<grid, NT_TC, SMEM_TOTAL, st>>>(a);
  return check_launch("dstcn_tc_kernel");
}

}  // namespace wekws
