// Streaming CTC keyword spotter on the device: wekws/bin/stream_kws_ctc.py:218-529 (KeyWordSpotter) for many streams.
//   kws_splice_kernel    accept_wave :346-364  -- the PCM carried from the last chunk in front of the new samples
//                        (a ragged staging buffer the Fbank kernel reads with per-stream lengths) + the new carry
//   kws_context_kernel   accept_wave :366-397  -- context expansion with the carried feature rows, then frame skip
//                        with the carried offset, rows packed back to back for the model
//   kws_detect_kernel    forward :489-512 -- per row one streaming beam step (ctc_beam.cuh) followed by
//                        execute_detection :411-480, stop after an activation, the end-of-chunk max_frames reset
//   kws_reset_kernel     reset :516-519 / the decoder half of reset_all :521-529
// Every row count and offset is planned on the host from sample counts it already knows (wekws_b200/spotter.py), so
// nothing is read back to plan a call.
#include <math.h>

#include "common.cuh"
#include "ctc_beam.cuh"

namespace wekws {
namespace {

using namespace beam;

// Persistent per-stream decoder + detector state (global memory).  It keeps only what survives a chunk: the pruned
// hypotheses and their node pool (the transient next_hyps of beam::Work stay in shared memory), ~19 KB per stream
// instead of the 44 KB of a full Work.
struct KwsState {
  Hyp cur[PBM];
  int32_t nframe[POOLM];
  float nprob[POOLM];
  int16_t ntok[POOLM];
  int32_t ncur, npool, overflow, pad_;
  double hit_score;             // self.hit_score: compounds over frames, only reset() sets it back to 1.0
  long long total_frames;       // self.total_frames
  long long last_active_pos;    // self.last_active_pos (-1 = never activated)
};

__device__ __forceinline__ void state_reset(KwsState& s, bool full) {
  s.ncur = 1; s.npool = 0;
  s.cur[0].pb = 1.0; s.cur[0].pnb = 0.0; s.cur[0].len = 0; s.cur[0].nlen = 0;
  s.hit_score = 1.0;
  if (full) { s.total_frames = 0; s.last_active_pos = -1; s.overflow = 0; }
}

__global__ void kws_reset_kernel(KwsState* __restrict__ st, const int32_t* __restrict__ ids, long long n, int full) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  state_reset(st[ids ? ids[i] : i], full != 0);
}

struct DetectArgs {
  const float* probs;           // (R, V) rows of all streams back to back
  const int32_t* row_off;       // (B) first row of stream b
  const int32_t* rows;          // (B) rows of stream b this call (0: nothing runs, result state -1)
  long long B;
  int V;
  const int32_t* allowed;       // keywords_idxset
  int n_allowed;
  const int32_t* kw_tokens;     // keyword k = kw_tokens[kw_off[k] .. kw_off[k+1])
  const int32_t* kw_off;
  int nkw;
  wekws_kws_config cfg;
  KwsState* state;
  int64_t* result;              // (B, WEKWS_KWS_RESULT_FIELDS)
};

// execute_detection (:411-480) on the current hypotheses; returns 1 on activation
__device__ int detect(const Work& w, const DetectArgs& a, double& hit_score, long long& last_active_pos, int& kw,
                      int& start, int& end) {
  int hit = -1;
  start = 0; end = 0;
  for (int h = 0; h < w.ncur && hit < 0; ++h) {
    const Hyp& c = w.cur[h];
    for (int k = 0; k < a.nkw; ++k) {
      const int nl = a.kw_off[k + 1] - a.kw_off[k];
      const int off = is_sublist(c.tok, c.len, a.kw_tokens + a.kw_off[k], nl);
      if (off != -1) {
        hit = k;
        start = w.nframe[c.node[off]];
        end = w.nframe[c.node[off + nl - 1]];
        for (int i = off; i < off + nl; ++i) hit_score = __dmul_rn(hit_score, (double)w.nprob[c.node[i]]);
        break;
      }
    }
    if (hit >= 0) hit_score = sqrt(hit_score);
  }
  const int duration = end - start;
  kw = hit;
  if (hit >= 0 && hit_score >= a.cfg.threshold && a.cfg.min_frames <= duration && duration <= a.cfg.max_frames &&
      (last_active_pos == -1 || end - last_active_pos >= a.cfg.interval_frames)) {
    last_active_pos = end;
    return 1;
  }
  return 0;
}

__global__ void __launch_bounds__(32) kws_detect_kernel(const DetectArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  Work& w = *reinterpret_cast<Work*>(smem);
  uint32_t* allow = reinterpret_cast<uint32_t*>(smem + sizeof(Work));
  const int lane = threadIdx.x;
  const long long b = blockIdx.x;
  const int n = a.rows[b];
  KwsState& st = a.state[b];
  int64_t* res = a.result + b * WEKWS_KWS_RESULT_FIELDS;
  if (n <= 0) {                                  // forward :484-485: no feature rows -> {} and nothing runs
    if (lane == 0) {
      res[0] = -1; res[1] = -1; res[2] = 0; res[3] = 0; res[4] = 0; res[5] = st.overflow;
    }
    return;
  }
  build_allow(allow, a.V, a.allowed, a.n_allowed, lane);
  if (lane == 0) {
    w.ncur = st.ncur; w.npool = st.npool; w.overflow = st.overflow;
    for (int h = 0; h < st.ncur; ++h) w.cur[h] = st.cur[h];
    for (int i = 0; i < st.npool; ++i) { w.ntok[i] = st.ntok[i]; w.nframe[i] = st.nframe[i]; w.nprob[i] = st.nprob[i]; }
  }
  __syncwarp();

  const int skip = a.cfg.frame_skip;
  const long long total = st.total_frames;
  double hit_score = st.hit_score;
  long long last_active_pos = st.last_active_pos;
  int activated = 0, kw = -1, start = 0, end = 0;
  const float* P = a.probs + (long long)a.row_off[b] * a.V;
  for (int t = 0; t < n; ++t) {
    int s_idx[SBM];
    float s_prob[SBM];
    const int ns = warp_topk_filter(P + (long long)t * a.V, a.V, a.cfg.score_beam, allow, lane, s_idx, s_prob);
    if (lane == 0) {
      if (ns > 0) advance(w, (int)(total + (long long)t * skip), s_idx, s_prob, ns, a.cfg.path_beam);
      // detection runs on every frame, also when the filter left the beam as it was (:160-161)
      activated = detect(w, a, hit_score, last_active_pos, kw, start, end);
    }
    activated = __shfl_sync(0xffffffffu, activated, 0);
    if (activated) break;                        // :495-501: reset(), the rest of the chunk is not decoded
  }

  if (lane == 0) {
    double score = hit_score;
    if (activated) { init_hyps(w); hit_score = 1.0; }
    const long long total_after = total + (long long)n * skip;        // :504, all rows, also after an activation
    // :509-512: drop a hypothesis whose first token is more than max_frames old
    if (w.ncur > 0 && w.cur[0].len > 0 && total_after - w.nframe[w.cur[0].node[0]] > a.cfg.max_frames) {
      init_hyps(w);
      hit_score = 1.0;
    }
    st.ncur = w.ncur; st.npool = w.npool; st.overflow = w.overflow;
    for (int h = 0; h < w.ncur; ++h) st.cur[h] = w.cur[h];
    for (int i = 0; i < w.npool; ++i) { st.ntok[i] = w.ntok[i]; st.nframe[i] = w.nframe[i]; st.nprob[i] = w.nprob[i]; }
    st.hit_score = hit_score;
    st.total_frames = total_after;
    st.last_active_pos = last_active_pos;
    res[0] = activated;
    res[1] = activated ? kw : -1;
    res[2] = activated ? start : 0;
    res[3] = activated ? end : 0;
    res[4] = activated ? __double_as_longlong(score) : 0;
    res[5] = w.overflow;
  }
}

// stage[b, i] = (carry ++ new)[i]; carry_out[b, i - consumed[b]] = the same sample (the tail the Fbank did not consume)
__global__ void kws_splice_kernel(const int16_t* __restrict__ pcm, long long pcm_stride, const int32_t* __restrict__ new_len,
                                  const int32_t* __restrict__ carry_len, const int32_t* __restrict__ consumed,
                                  const int16_t* __restrict__ carry_in, int16_t* __restrict__ carry_out, long long carry_cap,
                                  int16_t* __restrict__ stage, long long stage_stride) {
  const long long b = blockIdx.y;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int c = carry_len[b];
  if (i >= c + new_len[b]) return;
  const int16_t v = i < c ? carry_in[b * carry_cap + i] : pcm[b * pcm_stride + (i - c)];
  stage[b * stage_stride + i] = v;
  const long long j = i - consumed[b];
  if (j >= 0) carry_out[b * carry_cap + j] = v;
}

// One block per (output row, stream).  Expanded row i of stream b is ctx row r = off[b] + i * skip:
//   concat(pad[r], ..., pad[r + left + right]) with pad = left copies of feats[0] ++ feats on the first chunk
//   (fc_len < 0) and pad = carried rows ++ feats afterwards.  Without expansion the row is feats[r].
// Blocks i < left + right also write the next carry: the chunk's last min(left + right, nf) raw rows, or the old
// carry again when the stream produced no rows this call (the caller swaps fc_in / fc_out every call).
__global__ void kws_context_kernel(const float* __restrict__ feats, long long T, int D, const int32_t* __restrict__ nf,
                                   const float* __restrict__ fc_in, const int32_t* __restrict__ fc_len,
                                   float* __restrict__ fc_out, int left, int right, int expand, int skip,
                                   const int32_t* __restrict__ off, const int32_t* __restrict__ row_off,
                                   const int32_t* __restrict__ rows, float* __restrict__ out) {
  const long long b = blockIdx.y;
  const int i = blockIdx.x;
  const int W = expand ? left + right + 1 : 1, C = left + right;
  const float* f = feats + b * T * D;
  if (i < rows[b]) {
    const int r = off[b] + i * skip;
    const int c = fc_len[b];
    float* o = out + ((long long)row_off[b] + i) * W * D;
    for (int e = threadIdx.x; e < W * D; e += blockDim.x) {
      const int k = e / D, d = e - k * D, p = r + k;
      float v;
      if (!expand) v = f[(long long)r * D + d];
      else if (c < 0) v = f[(long long)(p < left ? 0 : p - left) * D + d];
      else v = p < c ? fc_in[(b * C + p) * D + d] : f[(long long)(p - c) * D + d];
      o[e] = v;
    }
  }
  if (expand && i < C) {
    const int n = nf[b], c = fc_len[b];
    if (n > 0) {
      const int cn = n < C ? n : C;
      if (i < cn)
        for (int d = threadIdx.x; d < D; d += blockDim.x) fc_out[(b * C + i) * D + d] = f[(long long)(n - cn + i) * D + d];
    } else if (i < c) {
      for (int d = threadIdx.x; d < D; d += blockDim.x) fc_out[(b * C + i) * D + d] = fc_in[(b * C + i) * D + d];
    }
  }
}

}  // namespace
}  // namespace wekws

using namespace wekws;

extern "C" int64_t wekws_kws_state_bytes(void) { return (int64_t)sizeof(KwsState); }

extern "C" int wekws_kws_reset(void* d_state, int64_t B, const int32_t* d_streams, int64_t n_streams, int full,
                               void* stream) {
  WEKWS_REQUIRE(B >= 0 && n_streams >= 0 && (d_streams || n_streams <= B), "wekws_kws_reset: bad sizes");
  const long long n = d_streams ? n_streams : B;
  if (n == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_state, "wekws_kws_reset: null state");
  kws_reset_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>((KwsState*)d_state, d_streams, n, full);
  return check_launch("kws_reset_kernel");
}

extern "C" int wekws_kws_detect(const float* d_probs, const int32_t* d_row_offsets, const int32_t* d_rows, int64_t B,
                                int V, const int32_t* d_token_set, int n_tokens, const int32_t* d_kw_tokens,
                                const int32_t* d_kw_offsets, int num_keywords, const wekws_kws_config* cfg,
                                void* d_state, int64_t* d_result, void* stream) {
  WEKWS_REQUIRE(cfg, "wekws_kws_detect: null config");
  WEKWS_REQUIRE(B >= 0 && V >= 1 && V <= 32767, "wekws_kws_detect: bad sizes (vocabulary <= 32767)");
  WEKWS_REQUIRE(cfg->score_beam >= 1 && cfg->score_beam <= WEKWS_CTC_MAX_SCORE_BEAM && cfg->score_beam <= V,
                "score_beam %d out of range (1..%d)", cfg->score_beam, WEKWS_CTC_MAX_SCORE_BEAM);
  WEKWS_REQUIRE(cfg->path_beam >= 1 && cfg->path_beam <= WEKWS_CTC_MAX_PATH_BEAM, "path_beam %d out of range (1..%d)",
                cfg->path_beam, WEKWS_CTC_MAX_PATH_BEAM);
  WEKWS_REQUIRE(cfg->frame_skip >= 1, "frame_skip must be >= 1");
  WEKWS_REQUIRE(num_keywords >= 1 && n_tokens >= 0, "wekws_kws_detect: at least one keyword is needed");
  if (B == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_row_offsets && d_rows && d_kw_tokens && d_kw_offsets && d_state && d_result &&
                    (n_tokens == 0 || d_token_set),
                "wekws_kws_detect: null argument");
  WEKWS_REQUIRE(B < (1ll << 31), "wekws_kws_detect: too many streams");
  DetectArgs a;
  a.probs = d_probs; a.row_off = d_row_offsets; a.rows = d_rows; a.B = B; a.V = V;
  a.allowed = d_token_set; a.n_allowed = n_tokens;
  a.kw_tokens = d_kw_tokens; a.kw_off = d_kw_offsets; a.nkw = num_keywords;
  a.cfg = *cfg; a.state = (KwsState*)d_state; a.result = d_result;
  const size_t smem = sizeof(Work) + (size_t)((V + 31) / 32) * 4;
  WEKWS_REQUIRE(smem <= 227 * 1024, "kws detect: vocabulary %d too large for the shared-memory token bitmap", V);
  static size_t attr_bytes[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_bytes[dev] < smem) {
    WEKWS_CUDA_OK(cudaFuncSetAttribute(kws_detect_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_bytes[dev] = smem;
  }
  kws_detect_kernel<<<(unsigned)B, 32, smem, (cudaStream_t)stream>>>(a);
  return check_launch("kws_detect_kernel");
}

extern "C" int wekws_kws_splice(const int16_t* d_pcm, int64_t pcm_stride, const int32_t* d_new_len,
                                const int32_t* d_carry_len, const int32_t* d_consumed, const int16_t* d_carry_in,
                                int16_t* d_carry_out, int64_t carry_cap, int16_t* d_stage, int64_t stage_stride,
                                int64_t B, void* stream) {
  WEKWS_REQUIRE(B >= 0 && pcm_stride >= 0 && carry_cap >= 0 && stage_stride >= 0, "wekws_kws_splice: bad sizes");
  if (B == 0 || stage_stride == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_new_len && d_carry_len && d_consumed && d_stage && (d_pcm || pcm_stride == 0) &&
                    (carry_cap == 0 || (d_carry_in && d_carry_out)),
                "wekws_kws_splice: null argument");
  WEKWS_REQUIRE(d_carry_in != d_carry_out || carry_cap == 0, "wekws_kws_splice: carry_in and carry_out must differ");
  WEKWS_REQUIRE(B < 65536, "wekws_kws_splice: more than 65535 streams in one call");
  dim3 grid((unsigned)((stage_stride + 255) / 256), (unsigned)B);
  kws_splice_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_pcm, pcm_stride, d_new_len, d_carry_len, d_consumed,
                                                            d_carry_in, d_carry_out, carry_cap, d_stage, stage_stride);
  return check_launch("kws_splice_kernel");
}

extern "C" int wekws_kws_context(const float* d_feats, int64_t B, int64_t T, int D, const int32_t* d_num_frames,
                                 const float* d_carry_in, const int32_t* d_carry_len, float* d_carry_out, int left,
                                 int right, int expand, int skip, const int32_t* d_skip_offset,
                                 const int32_t* d_row_offsets, const int32_t* d_rows, int64_t max_rows, float* d_out,
                                 void* stream) {
  WEKWS_REQUIRE(B >= 0 && T >= 0 && D >= 1 && left >= 0 && right >= 0 && skip >= 1 && max_rows >= 0,
                "wekws_kws_context: bad sizes");
  WEKWS_REQUIRE(!expand || left + right >= 1, "wekws_kws_context: context expansion needs left + right >= 1");
  const long long gx = expand && left + right > max_rows ? left + right : max_rows;
  if (B == 0 || gx == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_num_frames && d_carry_len && d_skip_offset && d_row_offsets && d_rows && (d_feats || T == 0) &&
                    (max_rows == 0 || d_out) && (!expand || (d_carry_in && d_carry_out && d_carry_in != d_carry_out)),
                "wekws_kws_context: null argument");
  WEKWS_REQUIRE(B < 65536 && gx < (1ll << 31), "wekws_kws_context: more than 65535 streams in one call");
  dim3 grid((unsigned)gx, (unsigned)B);
  kws_context_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(d_feats, T, D, d_num_frames, d_carry_in, d_carry_len,
                                                             d_carry_out, left, right, expand ? 1 : 0, skip,
                                                             d_skip_offset, d_row_offsets, d_rows, d_out);
  return check_launch("kws_context_kernel");
}
