// Tensor-core (tcgen05 / TMEM) fused MDTC forward for hidden_dim 64 -- the throughput path (round-2 layout).
//
// Same math as conv_backbone.cu (KWSModel.forward, reference wekws/model/kws_model.py:65-76 with
// mdtc.py:95-121 blocks, BatchNorm folded), but every dense GEMM (first Linear 80->64 and the 34
// pointwise 64x64 convolutions) runs on the 5th-gen tensor cores:
//   * bf16 "x3" operand split (tc_common.cuh): result within ~2^-16 of fp32 (posterior error ~1e-5, bar 1e-4);
//   * the A operand (activations) lives in TENSOR MEMORY: a thread writes its row with tcgen05.st, the MMA reads
//     it from TMEM (tcgen05.mma, A-from-TMEM form); B (weights) is a pre-swizzled K-major SWIZZLE_128B image in
//     shared memory, streamed by cp.async.bulk into a 2-slot ring;
//   * accumulators in TMEM, read back with tcgen05.ld.  Per tile: 64 columns D + 48 hi + 48 lo.
//
// One CTA per SM holds ALL of its streams (up to 7 x 40 frames) resident for the whole network.  What changed
// against round 1 (2025 warp-instructions per frame, every warp in the same phase at the same time):
//   * the residual stream is CHANNEL-MINOR: X[col][64 ch] (256 B per frame column, every stream's cache slice in the
//     columns directly in front of its frames, so a dilated tap is a column offset), 16-byte chunks XOR-swizzled
//     by (col & 7) -- a thread reads 8 channels of a tap with two conflict-free LDS.128 instead of 8 LDS.32;
//   * a thread owns a whole ROW (all 64 channels of one frame): 4 warps = one 128-row tile = one GROUP, and the
//     three groups run the network independently of each other (own mbarriers, a 128-thread named barrier per
//     block, own MMA-issue warp), so the CUDA-core phases of one tile overlap the tensor-core phases of the others
//     without any CTA-wide lock step;
//   * depthwise taps and bias adds use packed fma.rn.f32x2 / add.rn.f32x2; the ReLU of the pointwise-1 epilogue is
//     folded into the bf16 split (cvt.rz.relu / cvt.rn.relu), the split itself is 5 instructions per pair;
//   * each group stores its new cache slices while its own pointwise-1 GEMM runs.
//
// 15 warps: 12 compute (group g = warp / 4, TMEM lane quarter q = warp % 4; lane 0 of a group's first warp issues the
// group's MMAs once the other three warps have arrived), 1 weight / vector ring warp, 2 loaders (cache slices by 2-D
// TMA tensor copies into landing slots, transposed into X).
#include <stdlib.h>

#include "common.cuh"
#include "mdtc_tc.h"
#include "tc_common.cuh"

// per-phase cycle counters of a few warps (debug builds with -DMDTC_TIMING=1 only; see profiles/r02_mdtc_notes.md)
#ifndef MDTC_TIMING
#define MDTC_TIMING 0
#endif
#if MDTC_TIMING
#define TPH(acc) { const long long t_now_ = clock64(); acc += t_now_ - t_last_; t_last_ = t_now_; }
#else
#define TPH(acc)
#endif

namespace wekws {

namespace {

using namespace tc;

constexpr int NG = 3;                      // row tiles in flight == compute groups
constexpr int NCG = 2;                     // threads per row: thread (q, g) owns channels [32 g, 32 g + 32) of row 32 q + lane
constexpr int WPG = 4 * NCG;               // warps per group (tile)
constexpr int NCW = NG * WPG;              // compute warps (24)
constexpr int W_WGT = NCW;                 // warp 24: weight / vector ring
constexpr int W_LD = W_WGT + 1;            // warps 25..27: cache loaders, one per tile
constexpr int NT_TC = (W_LD + NG) * 32;    // 896 threads: 7 warps per scheduler -> 72 registers per thread
constexpr int C = 64;
constexpr int XCOLS = 504;                 // frame columns of X (n_streams * Lw <= XCOLS)
constexpr int X_BYTES = XCOLS * 256;       // 129024: X[col][64] fp32
constexpr int STG_FLOATS = 64 * 32;        // TMA landing slot: one stream's cache slice [64][pad <= 32]
constexpr int NSLOT = 7;                   // TMA landing slots, shared out among the tiles' loaders by stream count
constexpr int W_SLOT = 16384;              // hi + lo image of one 64x64 matrix
constexpr int OFF_X = 0;
constexpr int OFF_STG = OFF_X + X_BYTES;                   // 129024
constexpr int OFF_W = OFF_STG + NSLOT * STG_FLOATS * 4;    // 186368 (1024-aligned: SWIZZLE_128B images)
constexpr int OFF_END = OFF_W + 2 * W_SLOT;                // 219136
constexpr int SMEM_TOTAL = OFF_END + 1024;                 // incl. alignment slack
static_assert(OFF_W % 1024 == 0, "weight images must be 1024-byte aligned");
static_assert(SMEM_TOTAL <= 232448, "exceeds the 227 KB of shared memory a CTA may use");
// TMEM columns of tile i: [160 i, 160 i + 64) accumulator, + 64.. A hi (<= 48 cols = K 96), + 112.. A lo
constexpr int TM_TILE = 160, TM_AHI = 64, TM_ALO = 112, TM_COLS = 512;

__device__ __forceinline__ void group_barrier(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(32 * WPG) : "memory"); }
// Layout of X: frame column col holds its 64 channels in 256 bytes; the 16-byte chunk with channels 8m..8m+3 sits at
// chunk (m ^ (col & 7)) of the first 128 bytes, channels 8m+4..8m+7 at the same chunk of the second 128 bytes:
//   address(col, 8m + 4h + u) = xs + ((col << 8) | ((col & 7) << 4)) ^ (m << 4)  +  128 h  +  4 u
// 2-D TMA tensor copy global -> shared (box given by the tensor map), completion on an mbarrier
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}


// The service roles are separate NON-INLINED functions on purpose: compiled on their own they do not compete with the
// compute groups for uniform registers, which is what lets ptxas keep the per-block tap / bias constants of the
// compute code in the uniform datapath (LDCU + FFMA2 / FADD2 with UR operands) instead of vector LDC loads.
struct Bars {
  uint64_t *mma_bar, *halo_bar, *a_rdy, *h_free, *w_bar, *w_free, *vec_bar, *stg_bar;
};

// WEIGHT / VECTOR RING (one thread): slot 0 carries Linear atom 0, W1(0), W1(1), ...; slot 1 [Linear atom 1], W2(0), ...
__device__ __noinline__ void weights_role(const TcArgs& a, uint8_t* base, Bars B, int K, int natoms, uint32_t& wf_par,
                                          bool first_pass) {
  uint8_t* Wslot[2] = {base + OFF_W, base + OFF_W + W_SLOT};
  auto load_w = [&](int slot, const uint8_t* src) {
    mbar_arrive_expect_tx(&B.w_bar[slot], W_SLOT);
    bulk_g2s(Wslot[slot], src, W_SLOT, &B.w_bar[slot]);
  };
  auto wait_free = [&](int slot) {             // every tile's MMAs on the slot's current weights are done
    mbar_wait_backoff(&B.w_free[slot], (wf_par >> slot) & 1);
    wf_par ^= 1u << slot;
  };
  load_w(0, a.wimg);
  if (natoms > 1) load_w(1, a.wimg + W_SLOT);
  for (int b = 0; b <= a.nblocks; ++b) {
    const uint8_t* wb = a.wimg + (size_t)(2 + 2 * b) * W_SLOT;
    wait_free(0);
    if (b < a.nblocks) load_w(0, wb);
    if (b > 0 || natoms > 1) wait_free(1);
    if (b < a.nblocks) load_w(1, wb + W_SLOT);
  }
}

// LOADER WARP i serves tile i only: per (block, stream of the tile) one 2-D TMA copy [64][pad] into a landing slot,
// then the warp transposes it into the pad columns in front of the stream's frames in X.  A dedicated loader per tile
// means a group never queues behind another tile's slices (the round-2 profile showed the groups waiting 14 % of the
// time on halo_bar with two loaders walking the tiles in order).  The tile's ring of `nsl` landing slots is refilled
// the moment a slot is drained, i.e. the copy for the same stream of the NEXT block is in flight a whole block ahead.
__device__ __noinline__ void loader_role(const TcArgs& a, uint8_t* base, Bars B, int i, int lane, int K, int ns, int b0,
                                         int ntile, uint32_t& hf_par) {
  if (i >= ntile) return;
  float* STG = reinterpret_cast<float*>(base + OFF_STG);
  const uint32_t xs = smem_u32(base) + OFF_X;
  const int T = a.T, PADR = a.padr, Lw = a.padr + T, spt = a.spt;
  const int nst = min(spt, ns - i * spt), sg0 = i * spt;          // my streams: sg0 .. sg0 + nst
  const int njobs = a.nblocks * nst;
  const bool have_cache = a.in_cache != nullptr;
  // landing slots of tile t: the streams' share of the NSLOT slots (each tile at least one; ns <= NSLOT: one per stream)
  int slot0 = 0, nsl = 1;
  {
    int used = 0;
    for (int t = 0; t < ntile; ++t) {
      const int n_t = min(spt, ns - t * spt);
      int want = ns <= NSLOT ? n_t : max(1, (NSLOT * n_t) / ns);
      const int left = NSLOT - used - (ntile - 1 - t);               // keep one slot for every later tile
      if (want > left) want = left;
      if (t == i) { slot0 = used; nsl = want; }
      used += want;
    }
  }
  auto issue_tma = [&](int k) {                    // lane 0; job k = (blk, my m-th stream)
    const int blk = k / nst, sg = sg0 + (k - blk * nst);
    const int pad = a.dil[blk] * (K - 1);
    const uint32_t slot = slot0 + (uint32_t)k % nsl;
    mbar_arrive_expect_tx(&B.stg_bar[slot], (uint32_t)(C * pad * 4));
    tma_load_2d(STG + slot * STG_FLOATS, &a.tmap[a.tmap_idx[blk]], a.coff[blk], (b0 + sg) * C, &B.stg_bar[slot]);
  };
  // (an up-front cp.async.bulk.prefetch.L2 of the streams' whole cache rows was measured: 3 % slower)
  if (have_cache && lane == 0)
    for (int k0 = 0; k0 < nsl && k0 < njobs; ++k0) issue_tma(k0);
  int k = 0;
#if MDTC_TIMING
  long long t_hf = 0, t_stg = 0, t_tr = 0;
  long long t_last_ = clock64();
#endif
  for (int blk = 0; blk < a.nblocks; ++blk) {
    const int pad = a.dil[blk] * (K - 1);
    // X's pad columns of the tile are free once the depthwise conv of blk-1 is done (at blk 0: from the start)
    if (blk > 0) {
      if (lane == 0) mbar_wait_backoff(&B.h_free[i], hf_par & 1);
      hf_par ^= 1u;
      __syncwarp();
    }
    TPH(t_hf)
    // one 4-channel x 4-column item: four LDS.128 along the slot's (time-minor) channel rows, a register transpose,
    // four STS.128 (4 channels of one column each) -- 8 shared-memory instructions per 64 bytes
    const int lgg = 31 - __clz(pad >> 2);          // column groups of 4 per channel row (pad is a power of two >= 4)
    auto move_item = [&](const float* slotp, int colb, int r) {
      const int cq = r >> lgg, jg = r & ((1 << lgg) - 1);
      const float4* s4 = reinterpret_cast<const float4*>(slotp + 4 * cq * pad + 4 * jg);
      const float4 r0 = s4[0], r1 = s4[pad >> 2], r2 = s4[2 * (pad >> 2)], r3 = s4[3 * (pad >> 2)];
      const uint32_t sw = ((uint32_t)(cq >> 1) << 4), hi = (uint32_t)(cq & 1) * 128u;
      uint32_t col = (uint32_t)(colb + 4 * jg);
      sts_2x2(((xs + (col << 8) + ((col & 7u) << 4)) ^ sw) + hi, pack2(r0.x, r1.x), pack2(r2.x, r3.x)); ++col;
      sts_2x2(((xs + (col << 8) + ((col & 7u) << 4)) ^ sw) + hi, pack2(r0.y, r1.y), pack2(r2.y, r3.y)); ++col;
      sts_2x2(((xs + (col << 8) + ((col & 7u) << 4)) ^ sw) + hi, pack2(r0.z, r1.z), pack2(r2.z, r3.z)); ++col;
      sts_2x2(((xs + (col << 8) + ((col & 7u) << 4)) ^ sw) + hi, pack2(r0.w, r1.w), pack2(r2.w, r3.w));
    };
    if (have_cache && nsl >= nst) {
      // every stream of the tile has its own landing slot: wait for all of them (they were requested a block ago), move
      // everything in ONE flat loop, signal the group, and only then recycle the slots -- one latency chain per block
      // instead of one per stream (the per-stream version kept the group waiting on halo_bar 10-17 % of the time)
      for (int m = 0; m < nst; ++m) {
        const uint32_t use = (uint32_t)(k + m);
        mbar_wait(&B.stg_bar[slot0 + use % nsl], (use / nsl) & 1);
      }
      TPH(t_stg)
      const int per = 16 << lgg;
      for (int it = lane; it < nst * per; it += 32) {
        const int m = it >> (4 + lgg);
        move_item(STG + (slot0 + (uint32_t)(k + m) % nsl) * STG_FLOATS, (sg0 + m) * Lw + PADR - pad, it & (per - 1));
      }
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&B.halo_bar[i]);               // the tile's slices of this block are in place
        fence_proxy_async();                       // the slots were read through the generic proxy; TMA rewrites them
        for (int m = 0; m < nst; ++m)
          if (k + m + nsl < njobs) issue_tma(k + m + nsl);
      }
      k += nst;
      TPH(t_tr)
      continue;
    }
    for (int sg = sg0; sg < sg0 + nst; ++sg, ++k) {
      const int colb = sg * Lw + PADR - pad;       // first cache column of this stream for this block
      if (have_cache) {
        const uint32_t use = (uint32_t)k, slot = slot0 + use % nsl;
        if (lane == 0) mbar_wait_backoff(&B.stg_bar[slot], (use / nsl) & 1);
        __syncwarp();
        const float* slotp = STG + slot * STG_FLOATS;
        for (int it = lane; it < (16 << lgg); it += 32) move_item(slotp, colb, it);
        __syncwarp();                              // every lane has read the slot
        if (lane == 0 && k + nsl < njobs) {        // refill it: the same ring position, nsl jobs ahead
          fence_proxy_async();                     // the slot was read through the generic proxy; TMA rewrites it
          issue_tma(k + nsl);
        }
      } else {
        const f32x2 z = 0ull;
        for (int e = lane; e < pad * 16; e += 32) sts_2x2(xs + ((uint32_t)colb << 8) + 16u * (uint32_t)e, z, z);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&B.halo_bar[i]);    // the tile's slices of this block are in place
    TPH(t_tr)
  }
#if MDTC_TIMING
  if (blockIdx.x == 0 && lane == 0) printf("loader %d: wait h_free %lld, wait landing %lld, transposes %lld (nsl %d)\n", i, t_hf, t_stg, t_tr, nsl);
#endif
  // DW of the last block still signals h_free: consume it so the parity stays in step
  if (lane == 0) mbar_wait_backoff(&B.h_free[i], hf_par & 1);
  hf_par ^= 1u;
}

// KT: compile-time tap count (5 = every shipped mdtc config; 0 = read a.ktaps, taps guarded one by one)
template <int KT>
__global__ void __launch_bounds__(NT_TC, 1) mdtc_tc_kernel(const __grid_constant__ TcArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* base = smem_raw + ((1024 - (smem_u32(smem_raw) & 1023)) & 1023);
  __shared__ uint64_t mma_bar[NG], halo_bar[NG], a_rdy[NG], h_free[NG];
  __shared__ uint64_t w_bar[2], w_free[2], vec_bar[2], stg_bar[NSLOT];
  __shared__ uint64_t dw_tok[NG];                  // depthwise-phase token: passed group -> group (see the conv below)
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);   // warp-uniform for the compiler too (no divergence regions around the roles)
  const int T = a.T, K = KT ? KT : a.ktaps;
  const float* vec = a.vec;

  uint32_t sbase;                                  // shared-window address of `base`, pinned in a register
  asm volatile("mov.u32 %0, %1;" : "=r"(sbase) : "r"(smem_u32(base)));
  const uint32_t xs = sbase + OFF_X;

  if (tid == 0) {
    for (int i = 0; i < NG; ++i) {
      mbar_init(&mma_bar[i], 1); mbar_init(&halo_bar[i], 1); mbar_init(&a_rdy[i], WPG - 1); mbar_init(&h_free[i], WPG);
      mbar_init(&dw_tok[i], WPG);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&w_bar[i], 1); mbar_init(&w_free[i], NG); mbar_init(&vec_bar[i], 1); }
    mbar_fence_init();
  }
  if (warp == W_WGT) tmem_alloc(&tmem_slot, TM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = uniform32(tmem_slot);        // warp-uniform: MMA operands are then built in uniform registers
  const Bars bars{mma_bar, halo_bar, a_rdy, h_free, w_bar, w_free, vec_bar, stg_bar};
  // phase parities: every waiter keeps its own copy; all copies of a barrier advance in lock step
  uint32_t mma_par = 0, halo_par = 0, ar_par = 0, tok_par = 0;       // compute groups
  uint32_t hf_par = 0;                                               // loaders: bit i = tile i
  uint32_t w_par = 0, wf_par = 0;                                    // bit s = slot s
  const uint32_t idesc = make_idesc_bf16(128, 64);
  const int natoms = (a.idim + 63) / 64;
  const int PADR = a.padr, Lw = a.padr + T;
  const int spt = a.spt;                                             // streams per tile

  // balanced contiguous partition of the streams over the grid
  const int sb = (int)(((long long)a.B * blockIdx.x) / gridDim.x);
  const int se = (int)(((long long)a.B * (blockIdx.x + 1)) / gridDim.x);
  int done = sb;

  while (done < se) {
    const int remaining = se - done;
    const int passes_left = (remaining + a.smax - 1) / a.smax;
    const int ns = (remaining + passes_left - 1) / passes_left;      // streams of this pass (resident in X)
    const int b0 = done;
    done += ns;
    const int ntile = (ns + spt - 1) / spt;
    auto tile_streams = [&](int i) { return min(spt, ns - i * spt); };  // streams of tile i (sequential fill)

    // the landing slots are dealt out per pass (by stream count): their barriers start every pass from phase 0
    if (tid == 0) {
      for (int i = 0; i < NSLOT; ++i) mbar_init(&stg_bar[i], 1);
      mbar_fence_init();
    }
    __syncthreads();
    if (warp < NCW) {
      // ================================================================== COMPUTE GROUPS (WPG warps per tile)
      // warp = grp * WPG + 4 g + q: q = warp % 4 is the TMEM lane quarter the hardware lets this warp touch
      const int grp = warp / WPG, q = warp & 3, g = (warp % WPG) >> 2, wq = warp % WPG, row = 32 * q + lane;
      if (grp < ntile) {
        const int nst = tile_streams(grp), rows = nst * T;
        const bool live = row < rows, q_live = 32 * q < rows;
        const int s = live ? row / T : 0, tt = live ? row - s * T : 0;
        const int sg = grp * spt + s;                      // stream index inside the pass
        const int col = sg * Lw + PADR + tt;               // this row's frame column (dead rows alias a valid one)
        const uint32_t t_own = xs + ((uint32_t)col << 8) + (((uint32_t)col & 7u) << 4);
        const uint32_t tm_row = tmem + ((uint32_t)(32 * q) << 16) + TM_TILE * grp;
        float part[8];                                     // classifier partial sums of this row
#pragma unroll
        for (int j = 0; j < 8; ++j) part[j] = 0.f;

        // MMA issue (lane 0 of the group's first warp): 3-pass bf16x3 GEMM D (+)= A * W^T, A from TMEM (8 packed
        // columns per K step), W image in shared memory
        uint64_t dW_hi[2], dW_lo[2];
#pragma unroll
        for (int sl = 0; sl < 2; ++sl) {
          dW_hi[sl] = make_sdesc_sw128(sbase + OFF_W + sl * W_SLOT);
          dW_lo[sl] = make_sdesc_sw128(sbase + OFF_W + sl * W_SLOT + 8192);
        }
        const uint32_t dcol = tmem + TM_TILE * grp;
        auto issue_gemm = [&](int a_col, int slot, int ksteps, uint32_t& acc) {
          const uint32_t ahi = dcol + TM_AHI + a_col, alo = dcol + TM_ALO + a_col;
          for (int k = 0; k < ksteps; ++k) { umma_bf16_ts(dcol, ahi + 8 * k, dW_hi[slot] + 2 * k, idesc, acc); acc = 1; }
          for (int k = 0; k < ksteps; ++k) umma_bf16_ts(dcol, alo + 8 * k, dW_hi[slot] + 2 * k, idesc, 1);
          for (int k = 0; k < ksteps; ++k) umma_bf16_ts(dcol, ahi + 8 * k, dW_lo[slot] + 2 * k, idesc, 1);
        };
        // this warp's rows of the operand are in TMEM: the tile's other warps arrive and move on, the issuing warp waits
        // for them and dispatches GEMM `job` (-1: first Linear over slot 0 (+1); 0 / 1: the block's pointwise-1 / conv2
        // GEMM over that slot).  The two GEMMs of a block are dispatched by DIFFERENT warps (the last lane quarter of
        // each channel half -- the warps with the fewest live rows in a partly filled tile): a dispatch costs ~660
        // cycles, and with one warp doing both it was 1.3 k cycles behind its group at every block's barrier.
        auto hand_over = [&](int job) {
          const int issuer = job == 1 ? WPG - 1 : WPG / NCG - 1;
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (wq != issuer) {
            if (lane == 0) mbar_arrive(&a_rdy[grp]);
          } else {
            mbar_wait(&a_rdy[grp], ar_par);
            tc_fence_after();
            // the whole warp runs the issue path (uniform values -> descriptors in uniform registers, every MMA a single
            // instruction); only the tcgen05 instructions themselves are elected
            if (job < 0) {
              mbar_wait(&w_bar[0], w_par & 1);
              if (natoms > 1) mbar_wait(&w_bar[1], (w_par >> 1) & 1);
              if (elect_one_sync()) {
                uint32_t acc = 0;
                issue_gemm(0, 0, (min(a.idim, 64) + 15) >> 4, acc);
                if (natoms > 1) issue_gemm(32, 1, (a.idim - 64 + 15) >> 4, acc);
                umma_commit(&mma_bar[grp]);
                umma_commit(&w_free[0]);
                if (natoms > 1) umma_commit(&w_free[1]);
              }
            } else {
              mbar_wait(&w_bar[job], (w_par >> job) & 1);
              if (elect_one_sync()) {
                uint32_t acc = 0;
                issue_gemm(0, job, 4, acc);
                umma_commit(&mma_bar[grp]);
                umma_commit(&w_free[job]);      // the slot may be refilled once these MMAs are done
              }
            }
            __syncwarp();
          }
          ar_par ^= 1;                          // every warp keeps both phase counters: the issuer changes from GEMM to GEMM
          w_par ^= job < 0 ? (natoms > 1 ? 3u : 1u) : (1u << job);
        };
        auto wait_mma = [&]() {
          mbar_wait(&mma_bar[grp], mma_par);
          mma_par ^= 1;
          tc_fence_after();
        };

        // ---- features (+CMVN) -> bf16x3 operand rows in TMEM (8 K values = 4 packed columns per chunk)
        if (q_live) {
          const int nch = ((a.idim + 15) >> 4) * 2;        // 16-byte chunks incl. zero padding to a K step
          const float* src0 = a.feats + (size_t)(b0 + sg) * a.feat_bstride + (size_t)tt * a.idim;
          for (int ch = g; ch < nch; ch += NCG) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = 0.f;
            const int k0 = ch * 8;
            if (live && k0 < a.idim) {
              const float4 f0 = __ldg(reinterpret_cast<const float4*>(src0 + k0));
              const float4 f1 = __ldg(reinterpret_cast<const float4*>(src0 + k0) + 1);
              v[0] = f0.x; v[1] = f0.y; v[2] = f0.z; v[3] = f0.w; v[4] = f1.x; v[5] = f1.y; v[6] = f1.z; v[7] = f1.w;
              if (a.has_cmvn) {
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = (v[u] - __ldg(vec + a.v_mean + k0 + u)) * __ldg(vec + a.v_istd + k0 + u);
              }
            }
            uint32_t h[4], l[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) split_pair_rn(pack2(v[2 * u], v[2 * u + 1]), h[u], l[u]);
            tmem_st4(tm_row + TM_AHI + 4 * ch, h);
            tmem_st4(tm_row + TM_ALO + 4 * ch, l);
          }
        }
        hand_over(-1);
        // ---- x = relu(D + bp) -> X                                            (subsampling.py:53-57)
        wait_mma();
        if (q_live) {
          {
            const int half = g;
            uint32_t d[32];
            tmem_ld32_nowait(tm_row + 32 * half, d);
            tmem_ld_wait();
            const float4* bp = reinterpret_cast<const float4*>(vec + a.v_bp + 32 * half);
#pragma unroll
            for (int mm = 0; mm < 4; ++mm) {
              const float4 ba = __ldg(bp + 2 * mm), bb = __ldg(bp + 2 * mm + 1);
              auto E = [&](int u) { return __uint_as_float(d[8 * mm + u]); };
              const f32x2 o0 = pack2(fmaxf(E(0) + ba.x, 0.f), fmaxf(E(1) + ba.y, 0.f));
              const f32x2 o1 = pack2(fmaxf(E(2) + ba.z, 0.f), fmaxf(E(3) + ba.w, 0.f));
              const f32x2 o2 = pack2(fmaxf(E(4) + bb.x, 0.f), fmaxf(E(5) + bb.y, 0.f));
              const f32x2 o3 = pack2(fmaxf(E(6) + bb.z, 0.f), fmaxf(E(7) + bb.w, 0.f));
              const uint32_t ax = t_own ^ ((uint32_t)(4 * half + mm) << 4);
              if (live) { sts_2x2(ax, o0, o1); sts_2x2(ax + 128, o2, o3); }
            }
          }
        }
        tc_fence_before();
        group_barrier(grp);                  // X of the tile complete before the first depthwise conv reads across rows

        // ---- blocks
#if MDTC_TIMING
        long long t_halo = 0, t_dw = 0, t_ho0 = 0, t_cs = 0, t_w1 = 0, t_e1 = 0, t_ho1 = 0, t_w2 = 0, t_e2 = 0, t_gb = 0;
        long long t_last_ = clock64();
        const long long t_blocks0 = t_last_;
#endif
        for (int blk = 0; blk < a.nblocks; ++blk) {
          const int d = a.dil[blk], pad = d * (K - 1);
          const bool stack_end = (blk > 0) && (blk % a.stack_size == 0);
          // ---------------- depthwise dilated conv (+folded BN) -> operand rows in TMEM      (mdtc.py:56-57)
          mbar_wait(&halo_bar[grp], halo_par);
          halo_par ^= 1;
          TPH(t_halo)
          // The depthwise conv is the shared-memory-bandwidth phase (22 LDS.128 per 8 channels) while the epilogues and
          // the GEMM waits leave the load/store pipe idle.  Groups that run in lock step all hit it at once and then all
          // idle; a token handed from group to group (g -> g + 1 -> ... -> 0 of the next block) keeps exactly one
          // group in this phase, so the others' tensor-core and epilogue phases overlap it.
          const bool use_tok = ntile > 1 && (a.debug & 1);      // off by default: measured 9 % slower on B200 (profiles/r02_mdtc_notes.md)
          if (use_tok && !(blk == 0 && grp == 0)) {
            mbar_wait(&dw_tok[grp], tok_par);
            tok_par ^= 1;
          }
          if (q_live) {
            uint32_t tj[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) {
              const uint32_t cj = (uint32_t)(col - pad + j * d);
              tj[j] = xs + (cj << 8) + ((cj & 7u) << 4);
            }
#pragma unroll
            for (int mi = 0; mi < 8 / NCG; ++mi) {
              const int m = (8 / NCG) * g + mi;
              // (the folded depthwise bias is not added here: the host folds it through the pointwise-1 matrix into b1,
              // model_host.cu pack_tc -- it was 8 of the 48 LDS.128 per thread of this shared-memory-bound loop)
              f32x2 acc0 = 0ull, acc1 = 0ull, acc2 = 0ull, acc3 = 0ull;
#pragma unroll
              for (int j = 0; j < 5; ++j) {
                if (KT ? j < KT : j < K) {
                  const uint32_t aj = tj[j] ^ ((uint32_t)m << 4);
                  f32x2 x0, x1, x2, x3;
                  lds_2x2(aj, x0, x1);
                  lds_2x2(aj + 128, x2, x3);
                  const ulonglong2 wa = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * j + 2 * m]);       // LDCU
                  const ulonglong2 wb = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * j + 2 * m + 1]);
                  acc0 = fma2(x0, wa.x, acc0);
                  acc1 = fma2(x1, wa.y, acc1);
                  acc2 = fma2(x2, wb.x, acc2);
                  acc3 = fma2(x3, wb.y, acc3);
                }
              }
              uint32_t h[4], l[4];
              split_pair_rn(acc0, h[0], l[0]);
              split_pair_rn(acc1, h[1], l[1]);
              split_pair_rn(acc2, h[2], l[2]);
              split_pair_rn(acc3, h[3], l[3]);
              tmem_st4(tm_row + TM_AHI + 4 * m, h);
              tmem_st4(tm_row + TM_ALO + 4 * m, l);
            }
          }
          if (use_tok) {
            __syncwarp();
            if (lane == 0) mbar_arrive(&dw_tok[grp + 1 == ntile ? 0 : grp + 1]);
          }
          // this warp is done with the block's cache columns in front of the frames: when the new cache slice is made of
          // frame columns only (T >= pad) the loader may start transposing the next block's slices now, not after the
          // stores below (which read those columns when T < pad)
          const bool early_free = T >= pad;
          __syncwarp();
          if (early_free && lane == 0) mbar_arrive(&h_free[grp]);
          TPH(t_dw)
          hand_over(0);
          TPH(t_ho0)
          // ---------------- new cache slices of this tile while its pointwise-1 GEMM runs:
          // out_cache[b][c][off + j] = cat[c][T + j] (mdtc.py:113).  A warp reads 8 columns x 4 channels per request
          // (conflict-free in the swizzled layout); 8 lanes write 32 contiguous bytes of one cache row.
          {
            const int off = a.coff[blk];
            // lane -> (column j of the slice, channel-quad sub-index): one LDS.128 = 4 channels of one column, then four
            // stores, each lane-contiguous along a cache row (a 4x4 register-transposed variant with 16-byte stores was
            // measured: no faster, and it spills at 72 registers)
            const int jpl = pad < 32 ? pad : 32, lgj = 31 - __clz(jpl), qstep = 32 >> lgj;
            const int j = lane & (jpl - 1), qs = lane >> lgj, per = 16 >> (5 - lgj);      // quads passes per stream
            const int nitem = nst * per;
            for (int it = wq; it < nitem; it += WPG) {
              const int s2 = it / per, cq = (it - s2 * per) * qstep + qs;
              const int sg2 = grp * spt + s2;
              const uint32_t cc = (uint32_t)(sg2 * Lw + PADR + T - pad + j);
              const uint32_t src = ((xs + (cc << 8) + ((cc & 7u) << 4)) ^ ((uint32_t)(cq >> 1) << 4)) + (uint32_t)(cq & 1) * 128u;
              f32x2 v01, v23;
              lds_2x2(src, v01, v23);
              float v0, v1, v2, v3;
              unpack2(v01, v0, v1);
              unpack2(v23, v2, v3);
              float* g = a.out_cache + ((size_t)(b0 + sg2) * C + 4 * cq) * a.P + off + j;
              g[0] = v0; g[a.P] = v1; g[2 * a.P] = v2; g[3 * a.P] = v3;
            }
            if (!early_free) {
              __syncwarp();
              if (lane == 0) mbar_arrive(&h_free[grp]);    // the tile's cache columns may be overwritten
            }
          }
          // ---------------- h = relu(D + b1) -> operand rows in TMEM                          (mdtc.py:115)
          // (16 accumulator columns at a time: this thread's 32 channels in two rounds, 72 registers per thread)
          TPH(t_cs)
          wait_mma();
          TPH(t_w1)
          if (q_live) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              float dd[16];
              tmem_ld16(tm_row + 32 * g + 16 * hh, dd);
              uint32_t h[8], l[8];
#pragma unroll
              for (int mm = 0; mm < 2; ++mm) {
                const int m = 4 * g + 2 * hh + mm;
                const ulonglong2 ba = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * 5 + 2 * m]);      // b1
                const ulonglong2 bb = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * 5 + 2 * m + 1]);
                const float* e = dd + 8 * mm;
                split_pair_rz_relu(add2(pack2(e[0], e[1]), ba.x), h[4 * mm + 0], l[4 * mm + 0]);
                split_pair_rz_relu(add2(pack2(e[2], e[3]), ba.y), h[4 * mm + 1], l[4 * mm + 1]);
                split_pair_rz_relu(add2(pack2(e[4], e[5]), bb.x), h[4 * mm + 2], l[4 * mm + 2]);
                split_pair_rz_relu(add2(pack2(e[6], e[7]), bb.y), h[4 * mm + 3], l[4 * mm + 3]);
              }
              tmem_st8(tm_row + TM_AHI + 16 * g + 8 * hh, h);
              tmem_st8(tm_row + TM_ALO + 16 * g + 8 * hh, l);
            }
          }
          TPH(t_e1)
          hand_over(1);
          TPH(t_ho1)
          // ---------------- x' = relu(D + b2 + x) -> X; classifier partial sums at the end of a stack
          wait_mma();                                                          // (mdtc.py:116-118, 266-273)
          TPH(t_w2)
          if (q_live) {
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              float dd[16];
              tmem_ld16(tm_row + 32 * g + 16 * hh, dd);
#pragma unroll
              for (int mm = 0; mm < 2; ++mm) {
                const int m = 4 * g + 2 * hh + mm;
                const uint32_t ax = t_own ^ ((uint32_t)m << 4);
                const ulonglong2 ba = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * 6 + 2 * m]);                  // b2
                const ulonglong2 bb = *reinterpret_cast<const ulonglong2*>(&a.cw[blk][16 * 6 + 2 * m + 1]);
                f32x2 r0, r1, r2, r3;
                lds_2x2(ax, r0, r1);
                lds_2x2(ax + 128, r2, r3);
                const float* e = dd + 8 * mm;
                float o[8];
                unpack2(add2(add2(pack2(e[0], e[1]), ba.x), r0), o[0], o[1]);
                unpack2(add2(add2(pack2(e[2], e[3]), ba.y), r1), o[2], o[3]);
                unpack2(add2(add2(pack2(e[4], e[5]), bb.x), r2), o[4], o[5]);
                unpack2(add2(add2(pack2(e[6], e[7]), bb.y), r3), o[6], o[7]);
#pragma unroll
                for (int u = 0; u < 8; ++u) o[u] = fmaxf(o[u], 0.f);
                if (live) {
                  sts_2x2(ax, pack2(o[0], o[1]), pack2(o[2], o[3]));
                  sts_2x2(ax + 128, pack2(o[4], o[5]), pack2(o[6], o[7]));
                }
              }
            }
            if (stack_end) {
              // the classifier is linear: W_c (sum of stack outputs) = sum of W_c (stack output).  A compact loop over
              // the half row just written (own stores, program order) instead of unrolled copies inside the epilogue
#pragma unroll 1
              for (int mi = 0; mi < 8 / NCG; ++mi) {
                const int m = (8 / NCG) * g + mi;
                const uint32_t ax = t_own ^ ((uint32_t)m << 4);
                f32x2 r0, r1, r2, r3;
                lds_2x2(ax, r0, r1);
                lds_2x2(ax + 128, r2, r3);
                float o[8];
                unpack2(r0, o[0], o[1]); unpack2(r1, o[2], o[3]); unpack2(r2, o[4], o[5]); unpack2(r3, o[6], o[7]);
                const float* wc = vec + a.v_wc + (8 * m) * a.odim;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  if (j < a.odim) {
                    float p = part[j];
#pragma unroll
                    for (int u = 0; u < 8; ++u) p = fmaf(__ldg(wc + u * a.odim + j), o[u], p);
                    part[j] = p;
                  }
                }
              }
            }
          }
          TPH(t_e2)
          tc_fence_before();
          group_barrier(grp);                // x' of every row of the tile complete before the next block's conv
          TPH(t_gb)
        }
#if MDTC_TIMING
        if (blockIdx.x == 0 && lane == 0 && (warp == 0 || warp == 3 || warp == 7 || warp == 16))
          printf("warp %2d: blocks %lld cycles | halo %lld dw %lld handover0 %lld cache-store %lld wait1 %lld epi1 %lld handover1 %lld wait2 %lld epi2 %lld barrier %lld\n",
                 warp, clock64() - t_blocks0, t_halo, t_dw, t_ho0, t_cs, t_w1, t_e1, t_ho1, t_w2, t_e2, t_gb);
#endif

        if (ntile > 1 && (a.debug & 1) && grp == 0) {    // the last group's final hand-off: keep the parities in step
          mbar_wait(&dw_tok[0], tok_par);
          tok_par ^= 1;
        }
        // ---- classifier bias + activation: the g = 1 half parks its partial sums in the row's own (now dead) X column,
        // the g = 0 half adds them and writes the posterior
        if (NCG > 1) {
          if (g == 1 && live) {
            sts_2x2(t_own, pack2(part[0], part[1]), pack2(part[2], part[3]));
            sts_2x2(t_own + 128, pack2(part[4], part[5]), pack2(part[6], part[7]));
          }
          group_barrier(grp);
          if (g == 0 && live) {
            f32x2 p0, p1, p2, p3;
            lds_2x2(t_own, p0, p1);
            lds_2x2(t_own + 128, p2, p3);
            float o[8];
            unpack2(p0, o[0], o[1]); unpack2(p1, o[2], o[3]); unpack2(p2, o[4], o[5]); unpack2(p3, o[6], o[7]);
#pragma unroll
            for (int j = 0; j < 8; ++j) part[j] += o[j];
          }
        }
        if (live && g == 0) {
          float* o = a.out + (size_t)(b0 + sg) * a.out_bstride + (size_t)tt * a.odim;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (j < a.odim) {
              float y = part[j] + __ldg(vec + a.v_bc + j);
              if (a.act == WEKWS_ACT_SIGMOID) y = sigmoidf_acc(y);
              o[j] = y;
            }
          }
        }
      } else if (wq == 0) {
        // a group without streams in this pass still releases every weight slot use (w_free counts NG arrivals); all
        // lanes keep the same phase bookkeeping
        mbar_wait(&w_bar[0], w_par & 1);
        if (lane == 0) mbar_arrive(&w_free[0]);
        if (natoms > 1) {
          mbar_wait(&w_bar[1], (w_par >> 1) & 1);
          if (lane == 0) mbar_arrive(&w_free[1]);
        }
        w_par ^= natoms > 1 ? 3u : 1u;
        for (int blk = 0; blk < a.nblocks; ++blk)
          for (int job = 0; job < 2; ++job) {
            mbar_wait(&w_bar[job], (w_par >> job) & 1);
            w_par ^= 1u << job;
            if (lane == 0) mbar_arrive(&w_free[job]);
          }
      }
    } else if (warp == W_WGT) {
      if (lane == 0) weights_role(a, base, bars, K, natoms, wf_par, b0 == sb);
    } else {
      loader_role(a, base, bars, warp - W_LD, lane, K, ns, b0, ntile, hf_par);
    }
    __syncthreads();       // pass boundary: X, the landing slots and the rings are reused
  }

  tc_fence_before();
  __syncthreads();
  if (warp == W_WGT) tmem_dealloc(tmem, TM_COLS);
}

}  // namespace

bool tc_eligible(const TcArgs& a, int padmax) {
  if (a.idim % 8 != 0 || a.idim > 96 || a.odim > 8 || a.ktaps > 5) return false;   // A operand: 48 TMEM columns = K 96
  if (a.nblocks > kTcMaxBlocks) return false;                                        // taps / biases travel in the parameter block
  if (padmax > 32 || a.P % 4 != 0) return false;
  for (int b = 0; b < a.nblocks; ++b)
  {
    const int pad = a.dil[b] * (a.ktaps - 1);
    if (pad < 4 || (pad & (pad - 1)) != 0 || a.coff[b] % 4 != 0) return false;   // power-of-two slices, 16-byte aligned
  }
  return true;
}

int tc_max_T() { return 128; }

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
}  // namespace

int mdtc_tc_launch(TcArgs a, int padmax, cudaStream_t st) {
  WEKWS_REQUIRE(a.T >= 1 && a.T <= 128 && a.B >= 1, "mdtc_tc_launch: bad shape");
  a.padr = (padmax + 3) & ~3;
  const int Lw = a.padr + a.T;
  a.spt = 128 / a.T;                                   // streams per 128-row tile
  WEKWS_REQUIRE(a.spt >= 1 && Lw <= XCOLS, "mdtc_tc_launch: tile does not fit");
  int smax = NG * a.spt;                               // streams resident per pass
  if (smax > XCOLS / Lw) smax = XCOLS / Lw;
  a.smax = smax;
  {
    const char* dbg = getenv("WEKWS_TC_DEBUG");     // bit 0: depthwise-phase token on (A/B timing; results unchanged)
    a.debug = dbg ? atoi(dbg) : 0;
  }
  // tensor maps over the incoming cache (B*64 rows of P floats): one per distinct slice width
  if (a.in_cache != nullptr) {
    EncodeTiledFn enc = encode_tiled_fn();
    WEKWS_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled is not available from this driver");
    int pads[4], npads = 0;
    for (int b = 0; b < a.nblocks; ++b) {
      const int pad = a.dil[b] * (a.ktaps - 1);
      int i = 0;
      while (i < npads && pads[i] != pad) ++i;
      if (i == npads) {
        WEKWS_REQUIRE(npads < 4, "more than 4 distinct cache slice widths");
        pads[npads++] = pad;
        const cuuint64_t gdim[2] = {(cuuint64_t)a.P, (cuuint64_t)a.B * C};
        const cuuint64_t gstr[1] = {(cuuint64_t)a.P * sizeof(float)};
        const cuuint32_t box[2] = {(cuuint32_t)pad, (cuuint32_t)C};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult rc = enc(&a.tmap[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(a.in_cache), gdim,
                                gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        WEKWS_REQUIRE(rc == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d)", (int)rc);
      }
      a.tmap_idx[b] = i;
    }
  }
  const int sms = device_sm_count();
  const int grid = a.B < sms ? a.B : sms;
  static bool attr_set[64] = {false};
  if (int rc = set_max_dynamic_smem_once(attr_set, SMEM_TOTAL, mdtc_tc_kernel<5>, mdtc_tc_kernel<0>)) return rc;
  if (a.ktaps == 5) mdtc_tc_kernel<5><<<grid, NT_TC, SMEM_TOTAL, st>>>(a);
  else mdtc_tc_kernel<0><<<grid, NT_TC, SMEM_TOTAL, st>>>(a);
  return check_launch("mdtc_tc_kernel");
}

}  // namespace wekws
