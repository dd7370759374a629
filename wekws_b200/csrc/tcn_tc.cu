// Tensor-core (tcgen05 / TMEM) fused forward for the dense TCN backbone with hidden_dim 64
// (reference wekws/model/tcn.py:67-88 CnnBlock inside TCN :122-166; BatchNorm folded):
//     per block:  o = ReLU( sum_j W_j . cat(cache, x)[:, t + j*d] + b ) ;  x' = o + x
// i.e. a K-tap dilated convolution = K accumulating 64x64 GEMMs whose A operand is the residual stream
// shifted by j*d frames.  Same machinery as mdtc_tc.cu: all streams of a CTA resident in shared memory
// (X[c][col], cache slice in front of each stream's frames so a tap is a column offset), bf16x3 split,
// A operand written to TMEM row by row (tcgen05.st) into TWO alternating buffers per tile so the shifted
// copy of tap j+1 is produced while the MMAs of tap j run, accumulators in TMEM, weights as pre-swizzled
// 16 KB images streamed through a 4-slot ring by cp.async.bulk.  TCN cache rows are 105 floats and slices
// 7..56 floats wide -- not 16-byte multiples, so TMA cannot fetch them: the loader warps use 4-byte
// cp.async straight into X instead.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "tc_common.cuh"
#include "tcn_tc.h"

// per-phase cycle counters (debug builds with -DTCN_TIMING=1 only)
#ifndef TCN_TIMING
#define TCN_TIMING 0
#endif
#if TCN_TIMING
#define TPH(acc) { const long long t_now_ = clock64(); acc += t_now_ - t_last_; t_last_ = t_now_; }
#else
#define TPH(acc)
#endif

namespace wekws {

namespace {

using namespace tc;

constexpr int NCW = 16, NCT = NCW * 32, NT_TC = NCT + 96;
constexpr int C = 64;
constexpr int NTILE = 2;
constexpr int RPX = 512, XCOLS = 504;
constexpr int X_BYTES = 64 * RPX * 4;
constexpr int W_SLOT = 16384, NW = 4;
constexpr int OFF_X = 0, OFF_W = X_BYTES;
constexpr int SMEM_TOTAL = OFF_W + NW * W_SLOT + 1024;            // 197632
// TMEM columns of tile i (192 each): [0,64) accumulator; operand buffer b: hi at 64 + 64 b, lo at 96 + 64 b;
// the first Linear (K <= 96) uses hi at 64.., lo at 128..
constexpr int TM_TILE = 192, TM_COLS = 512;

__device__ __forceinline__ void compute_barrier() { asm volatile("bar.sync 1, %0;" ::"n"(NCT) : "memory"); }
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void split_to_tmem(const float (&v)[8], uint32_t t_hi, uint32_t t_lo) {
  uint32_t h[4], l[4];
  split2(v[0], v[1], h[0], l[0]); split2(v[2], v[3], h[1], l[1]);
  split2(v[4], v[5], h[2], l[2]); split2(v[6], v[7], h[3], l[3]);
  tmem_st4(t_hi, h);
  tmem_st4(t_lo, l);
}

__global__ void __launch_bounds__(NT_TC, 1) tcn_tc_kernel(const TcnTcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  __shared__ uint64_t mma_bar[NTILE], halo_bar[NTILE], a_rdy[NTILE][2], h_free[NTILE], ab_free[NTILE][2];
  __shared__ uint64_t w_bar[NW], w_free[NW];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_issuer = warp == NCW, is_loader = warp > NCW;
  const int q = warp & 3, g = (warp >> 2) & 3;
  const int row = 32 * q + lane;
  const int T = a.T, K = a.ktaps;
  const float* vec = a.vec;
  float* X = reinterpret_cast<float*>(base + OFF_X);
  uint8_t* Wring = base + OFF_W;
  uint32_t sbase;
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"(smem_u32(base)));

  if (tid == 0) {
    for (int i = 0; i < NTILE; ++i) {
      mbar_init(&mma_bar[i], 1); mbar_init(&halo_bar[i], 2); mbar_init(&a_rdy[i][0], NCW); mbar_init(&a_rdy[i][1], NCW);
      mbar_init(&h_free[i], NCW);
      mbar_init(&ab_free[i][0], 1); mbar_init(&ab_free[i][1], 1);
    }
    for (int i = 0; i < NW; ++i) { mbar_init(&w_bar[i], 1); mbar_init(&w_free[i], 1); }
    mbar_fence_init();
  }
#ifdef WEKWS_MBAR_WATCHDOG
  if (tid == 0 && blockIdx.x == 0)
    printf("tcn_tc barriers: mma_bar 0x%x halo_bar 0x%x a_rdy 0x%x h_free 0x%x ab_free 0x%x w_bar 0x%x w_free 0x%x\n",
           smem_u32(mma_bar), smem_u32(halo_bar), smem_u32(a_rdy), smem_u32(h_free), smem_u32(ab_free), smem_u32(w_bar),
           smem_u32(w_free));
#endif
  if (is_issuer) tmem_alloc(&tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform32(tmem_slot);      // warp-uniform: MMA operands are then built in uniform registers
  uint32_t mma_par = 0, halo_par = 0, ar_par = 0, hf_par = 0;
  uint32_t witem = 0;                              // issuer: weight items consumed so far (slot = item % NW)
  uint32_t ab_cnt[NTILE][2] = {{0, 0}, {0, 0}};     // compute: commits of ab_free[i][b] before the current block
  const uint32_t idesc = make_idesc_bf16(128, 64);
  const int natoms = (a.idim + 63) / 64;
  const int PADR = a.padr, Lw = a.padr + ((T + 3) & ~3);
  const int spt = a.spt;
  const int nitems = 2 + a.nblocks * K;             // weight images per pass: Wp atom 0, atom 1, then the taps

  const int sb = (int)(((long long)a.B * blockIdx.x) / gridDim.x);
  const int se = (int)(((long long)a.B * (blockIdx.x + 1)) / gridDim.x);
  int done = sb;

  while (done < se) {
    const int remaining = se - done;
    const int passes_left = (remaining + a.smax - 1) / a.smax;
    const int ns = (remaining + passes_left - 1) / passes_left;
    const int b0 = done;
    done += ns;
    const int ntile = (ns + spt - 1) / spt;
    auto tile_streams = [&](int i) { return min(spt, ns - i * spt); };

    if (is_issuer) {
      // ================================================================== MMA-ISSUE WARP
      // All lanes run the (uniform) control flow and descriptor arithmetic; the tcgen05 / bulk-copy instructions are
      // elected.  With `if (lane == 0)` around the whole role every MMA sat in an ELECT / R2UR waterfall loop.
      {
        int loaded = 0, freed = 0;                   // items whose load was issued / whose slot was reclaimed
        auto load_item = [&](int n) {                // item n of this pass -> its ring slot
          const uint32_t slot = (witem + (uint32_t)n) % NW;
          if (lane == 0) {
            mbar_arrive_expect_tx(&w_bar[slot], W_SLOT);
            bulk_g2s(Wring + slot * W_SLOT, a.wimg + (size_t)n * W_SLOT, W_SLOT, &w_bar[slot]);
          }
        };
        auto reclaim = [&](int n) {                  // wait until the MMAs that read item n are done, then refill
          const uint32_t use = witem + (uint32_t)n, slot = use % NW;
          mbar_wait(&w_free[slot], (use / NW) & 1);
          if (loaded < nitems) { load_item(loaded); ++loaded; }
        };
        auto wait_w = [&](int n) {
          const uint32_t use = witem + (uint32_t)n, slot = use % NW;
          mbar_wait(&w_bar[slot], (use / NW) & 1);
          return make_sdesc_sw128(smem_u32(Wring + slot * W_SLOT));
        };
        auto release_w = [&](int n) { if (elect_one_sync()) umma_commit(&w_free[(witem + (uint32_t)n) % NW]); };
        auto issue_gemm = [&](int i, int a_hi_col, int a_lo_col, uint64_t dwh, int ksteps, uint32_t& acc) {
          const uint32_t d = tmem + TM_TILE * i, ahi = d + a_hi_col, alo = d + a_lo_col;
          const uint64_t dwl = dwh + (8192 >> 4);
          if (elect_one_sync()) {
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, ahi + 8 * k, dwh + 2 * k, idesc, k == 0 ? acc : 1u);
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, alo + 8 * k, dwh + 2 * k, idesc, 1);
            for (int k = 0; k < ksteps; ++k) umma_bf16_ts(d, ahi + 8 * k, dwl + 2 * k, idesc, 1);
          }
          acc = 1;
        };
        // one hand-over barrier per operand buffer: with a single one the compute warps could complete the phase
        // of tap j+1 before this thread had observed the phase of tap j (their only back-pressure is ab_free of
        // tap j-1), and a parity wait cannot see a phase that is two behind
        auto wait_a = [&](int i, int b) {
          mbar_wait(&a_rdy[i][b], (ar_par >> (2 * i + b)) & 1);
          ar_par ^= 1u << (2 * i + b);
          tc_fence_after();
        };
        for (; loaded < NW && loaded < nitems; ++loaded) load_item(loaded);

        // ---- first Linear: items 0 (K columns 0..63) and 1 (64..)
        const int ks0 = (min(a.idim, 64) + 15) >> 4, ks1 = natoms > 1 ? (a.idim - 64 + 15) >> 4 : 0;
        const uint64_t dwp0 = wait_w(0), dwp1 = wait_w(1);
        for (int i = 0; i < ntile; ++i) {
          wait_a(i, 0);
          uint32_t acc = 0;
          issue_gemm(i, 64, 128, dwp0, ks0, acc);
          if (natoms > 1) issue_gemm(i, 64 + 32, 128 + 32, dwp1, ks1, acc);
          if (elect_one_sync()) umma_commit(&mma_bar[i]);
        }
        release_w(0); release_w(1);
        // ---- blocks: tap j of block blk is item 2 + blk*K + j
        for (int blk = 0; blk < a.nblocks; ++blk) {
          for (int j = 0; j < K; ++j) {
            const int n = 2 + blk * K + j;
            wd_mark(4000000 + n * 10);
            while (freed < n - 1) { reclaim(freed); ++freed; }      // slots of items consumed >= 2 taps ago
            const uint64_t dwh = wait_w(n);
            wd_mark(3000000 + n * 10);
            for (int i = 0; i < ntile; ++i) {
              wd_mark(1000000 + n * 10 + i);
              wait_a(i, j & 1);
              wd_mark(2000000 + n * 10 + i);
              uint32_t acc = j > 0 ? 1u : 0u;
              issue_gemm(i, 64 + 64 * (j & 1), 96 + 64 * (j & 1), dwh, 4, acc);
              if (elect_one_sync()) {
                umma_commit(&ab_free[i][j & 1]);
                if (j == K - 1) umma_commit(&mma_bar[i]);
              }
            }
            release_w(n);
          }
        }
        while (freed < nitems) { reclaim(freed); ++freed; }          // drain: keeps the ring parities in step
        witem += (uint32_t)nitems;
      }
    } else if (is_loader) {
      // (no loader role any more: the compute warps fetch the next block's cache slices themselves, see load_halo)
    } else {
      // ================================================================== COMPUTE WARPS
      int colx[NTILE], rows_i[NTILE];
#if TCN_TIMING
      long long t_halo = 0, t_abf = 0, t_stage = 0, t_ho = 0, t_cs = 0, t_wm = 0, t_epi = 0, t_bar = 0, t_last_ = 0;
#endif
#pragma unroll
      for (int i = 0; i < NTILE; ++i) {
        rows_i[i] = i < ntile ? tile_streams(i) * T : 0;
        const int s = row / T;
        colx[i] = row < rows_i[i] ? (i * spt + s) * Lw + PADR + (row - s * T) : XCOLS;
      }
      const bool q_live[NTILE] = {32 * q < rows_i[0], 32 * q < rows_i[1]};
      const uint32_t tm_row = tmem + ((uint32_t)(32 * q) << 16);
      const uint32_t xs = sbase + OFF_X;

      auto hand_over = [&](auto tc, int b) {
        constexpr int i = decltype(tc)::value;
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_rdy[i][b]);
      };
      auto wait_mma = [&](auto tc) {
        constexpr int i = decltype(tc)::value;
        mbar_wait(&mma_bar[i], (mma_par >> i) & 1);
        mma_par ^= 1u << i;
        tc_fence_after();
      };
      auto feat = [&](auto tc) {
        constexpr int i = decltype(tc)::value;
        if (q_live[i]) {
          const int nch = ((a.idim + 15) >> 4) * 2;
          const bool valid = row < rows_i[i];
          const int s = row / T, tt = row - s * T;
          const float* src0 = a.feats + (size_t)(b0 + i * spt + s) * a.feat_bstride + (size_t)tt * a.idim;
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
            split_to_tmem(v, tm_row + TM_TILE * i + 64 + 4 * ch, tm_row + TM_TILE * i + 128 + 4 * ch);
          }
        }
        hand_over(tc, 0);
      };
      auto epi0 = [&](auto tc) {                     // x = relu(D + bp) -> X
        constexpr int i = decltype(tc)::value;
        wait_mma(tc);
        if (!q_live[i]) return;
        float d[16];
        tmem_ld16(tm_row + TM_TILE * i + 16 * g, d);
        float* xp = X + (16 * g) * RPX + colx[i];
        const float4* bp = reinterpret_cast<const float4*>(vec + a.v_bp + 16 * g);
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          const float4 b = __ldg(bp + i4);
          xp[(4 * i4 + 0) * RPX] = fmaxf(d[4 * i4 + 0] + b.x, 0.f);
          xp[(4 * i4 + 1) * RPX] = fmaxf(d[4 * i4 + 1] + b.y, 0.f);
          xp[(4 * i4 + 2) * RPX] = fmaxf(d[4 * i4 + 2] + b.z, 0.f);
          xp[(4 * i4 + 3) * RPX] = fmaxf(d[4 * i4 + 3] + b.w, 0.f);
        }
      };
      // tap j of block blk: this thread's row of cat(cache, x) shifted by j*d frames -> operand buffer j & 1
      auto tap = [&](auto tc, int blk, int j, int d, int pad) {
        constexpr int i = decltype(tc)::value;
        const int b = j & 1;
        wd_mark(1000000 + blk * 1000 + j * 10 + i);
        // (the tile's cache slice is in place: load_halo + the barrier at the end of the previous block)
        if (j >= 2) {                                // the MMAs of tap j-2 have drained this buffer
          const uint32_t cidx = ab_cnt[i][b] + (uint32_t)(j >> 1) - 1u;
          mbar_wait(&ab_free[i][b], cidx & 1);
          tc_fence_after();
        }
        TPH(t_abf)
        wd_mark(3000000 + blk * 1000 + j * 10 + i);
        if (q_live[i]) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int cg = g + 4 * half;
            const uint32_t aj = xs + 4u * (uint32_t)(cg * 8 * RPX + colx[i] - pad + j * d);
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = lds_f32(aj + u * RPX * 4);
            split_to_tmem(v, tm_row + TM_TILE * i + 64 + 64 * b + 4 * cg, tm_row + TM_TILE * i + 96 + 64 * b + 4 * cg);
          }
        }
        TPH(t_stage)
        hand_over(tc, b);
        TPH(t_ho)
        wd_mark(4000000 + blk * 1000 + j * 10 + i);
      };
      // Cache slices of block `blk` -> the pad columns in front of every stream's frames, 4-byte cp.async (rows of the
      // cache are 105 floats, slices 7..56: nothing is 16-byte aligned), spread over ALL compute threads and issued one
      // block ahead, right after the last tap that reads the current block's slices -- the copies then overlap the last
      // tap, its GEMM and the epilogue; `halo_wait` + the block barrier publish them.  (Two dedicated loader warps with
      // a per-element division needed ~17 k cycles per block and the compute warps spent 55 % of their time waiting
      // for them: clock64 counters, profiles/r02_tcn_notes.md.)
      auto load_halo = [&](int blk) {
        const int pad = a.dil[blk] * (K - 1), off = a.coff[blk];
        const int per = C * pad;
        for (int e = tid; e < ns * per; e += NCT) {
          const int sg = e / per, r = e - sg * per, c = r / pad, p = r - c * pad;
          float* dst = X + c * RPX + sg * Lw + PADR - pad + p;
          if (a.in_cache) cp_async4(dst, a.in_cache + ((size_t)(b0 + sg) * C + c) * a.P + off + p);
          else *dst = 0.f;
        }
      };
      auto halo_wait = [&]() { asm volatile("cp.async.wait_all;\n" ::: "memory"); };
      // new cache slices (tcn.py:54); afterwards nobody reads the block's cache columns again
      auto store_cache = [&](int blk, int pad) {
        const int off = a.coff[blk];
        for (int i = 0; i < ntile; ++i) {
          const int nst = tile_streams(i), sg0 = i * spt, n = nst * C * pad;
          for (int e = tid; e < n; e += NCT) {
            const int cs = e / pad, j = e - cs * pad, s = cs >> 6, c = cs & 63;
            a.out_cache[((size_t)(b0 + sg0 + s) * C + c) * a.P + off + j] = X[c * RPX + (sg0 + s) * Lw + PADR - pad + T + j];
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&h_free[0]);
      };
      // every compute warp is past the taps (and cache stores) that read the current slices: the columns may be rewritten
      auto halo_free_wait = [&]() {
        mbar_wait(&h_free[0], hf_par & 1);
        hf_par ^= 1u;
      };
      // x' = relu(D + b) + x -> X                                          (tcn.py:60: no ReLU after the add)
      auto epi = [&](auto tc, int blk) {
        constexpr int i = decltype(tc)::value;
        const float* bb = vec + a.v_blocks + blk * a.v_blk_stride + 16 * g;
        wd_mark(5000000 + blk * 1000 + i);
        wait_mma(tc);
        TPH(t_wm)
        wd_mark(6000000 + blk * 1000 + i);
        if (!q_live[i]) return;
        float d[16];
        tmem_ld16(tm_row + TM_TILE * i + 16 * g, d);
        float* xp = X + (16 * g) * RPX + colx[i];
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(bb) + i4);
          const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int e = 4 * i4 + u;
            xp[e * RPX] = fmaxf(d[e] + bv[u], 0.f) + xp[e * RPX];
          }
        }
      };

      constexpr std::integral_constant<int, 0> T0{};
      constexpr std::integral_constant<int, 1> T1{};
      wd_mark(1);
      load_halo(0);                                  // overlaps the feature load and the first Linear
      feat(T0);
      if (ntile > 1) feat(T1);
      wd_mark(2);
      epi0(T0);
      if (ntile > 1) epi0(T1);
      wd_mark(3);
      halo_wait();
      tc_fence_before();
      compute_barrier();
      wd_mark(4);

#if TCN_TIMING
      t_last_ = clock64();
      const long long t_begin_ = t_last_;
#endif
      for (int blk = 0; blk < a.nblocks; ++blk) {
        const int d = a.dil[blk], pad = d * (K - 1);
        for (int j = 0; j < K; ++j) {
          // The last tap reads frames only (position t + pad), never the cache columns: store the new cache slices
          // and release the columns before it.  The stores then precede this warp's last hand-over, hence the last
          // GEMM and the epilogue (which overwrites x) cannot start before every warp's stores have been issued.
          if (j == K - 1) {
            store_cache(blk, pad);
            TPH(t_cs)
            halo_free_wait();
            if (blk + 1 < a.nblocks) load_halo(blk + 1);
            TPH(t_halo)
          }
          tap(T0, blk, j, d, pad);
          if (ntile > 1) tap(T1, blk, j, d, pad);
        }
#pragma unroll
        for (int i = 0; i < NTILE; ++i)
          if (i < ntile) { ab_cnt[i][0] += (uint32_t)((K + 1) >> 1); ab_cnt[i][1] += (uint32_t)(K >> 1); }
        epi(T0, blk);
        if (ntile > 1) epi(T1, blk);
        TPH(t_epi)
        halo_wait();
        tc_fence_before();
        compute_barrier();
        TPH(t_bar)
      }
#if TCN_TIMING
      if (blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 7))
        printf("tcn warp %d pass(ns=%d): blocks %lld cycles | halo %lld ab_free %lld staging %lld handover %lld cache-store %lld wait-mma %lld epilogue %lld barrier %lld\n",
               warp, ns, clock64() - t_begin_, t_halo, t_abf, t_stage, t_ho, t_cs, t_wm, t_epi, t_bar);
#endif

      // ---- classifier + activation on x (tcn.py:165 -> classifier.py:63-67)
      const int odim = a.odim;
      for (int i = 0; i < ntile; ++i) {
        const int nrow = tile_streams(i) * T;
        for (int idx = tid; idx < nrow * odim; idx += NCT) {
          const int r = idx / odim, j = idx - r * odim;
          const int s = r / T, tt = r - s * T;
          const float* xc = X + (i * spt + s) * Lw + PADR + tt;
          float y = __ldg(vec + a.v_bc + j);
#pragma unroll 8
          for (int c = 0; c < C; ++c) y = fmaf(__ldg(vec + a.v_wc + c * odim + j), xc[c * RPX], y);
          if (a.act == WEKWS_ACT_SIGMOID) y = sigmoidf_acc(y);
          a.out[(size_t)(b0 + i * spt + s) * a.out_bstride + (size_t)tt * odim + j] = y;
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

bool tcn_tc_eligible(const TcnTcArgs& a, int padmax) {
  if (a.idim % 8 != 0 || a.idim > 128 || a.odim > 8 || a.ktaps > 8 || a.ktaps < 2) return false;
  if (((padmax + 3) & ~3) + 8 > XCOLS) return false;
  return true;
}

int tcn_tc_max_T() { return 128; }

int tcn_tc_launch(TcnTcArgs a, int padmax, cudaStream_t st) {
  WEKWS_REQUIRE(a.T >= 1 && a.T <= 128 && a.B >= 1, "tcn_tc_launch: bad shape");
  a.padr = (padmax + 3) & ~3;
  const int Lw = a.padr + ((a.T + 3) & ~3);
  a.spt = 128 / a.T;
  WEKWS_REQUIRE(a.spt >= 1 && Lw <= XCOLS, "tcn_tc_launch: tile does not fit");
  int smax = NTILE * a.spt;
  if (smax > XCOLS / Lw) smax = XCOLS / Lw;
  a.smax = smax;
  const int sms = device_sm_count();
  const int grid = a.B < sms ? a.B : sms;
  static bool attr_set[64] = {false};
  if (int rc = set_max_dynamic_smem_once(attr_set, SMEM_TOTAL, tcn_tc_kernel)) return rc;
  tcn_tc_kernel<<<grid, NT_TC, SMEM_TOTAL, st>>>(a);
  return check_launch("tcn_tc_kernel");
}

}  // namespace wekws
