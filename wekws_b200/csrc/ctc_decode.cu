// CTC prefix beam search + keyword detection on the device (SURVEY 8f-2, CTC models): what the reference does per
// utterance / per frame in pure Python --
//   wekws/model/loss.py:206-312 ctc_prefix_beam_search (whole utterance, wekws/bin/score_ctc.py:198-200) and its
//   streaming twin wekws/bin/stream_kws_ctc.py:124-215 (one frame per call, hypotheses carried), followed by the
//   keyword look-up of score_ctc.py:201-220 / stream_kws_ctc.py:411-434 (is_sublist, sqrt of the product of the
//   token probabilities).
// The beam step itself (and the Python semantics it keeps bit-exactly) lives in ctc_beam.cuh, shared with the streaming
// keyword spotter of kws_stream.cu.
// One warp per utterance: all lanes scan the frame's V probabilities for the top score_beam entries, lane 0 runs the
// (tiny, inherently sequential) hypothesis update in shared memory.  Utterances are independent -> B warps.
#include <math.h>

#include "common.cuh"
#include "ctc_beam.cuh"
#include "ctc_decode.h"

namespace wekws {
namespace {

using namespace beam;

__global__ void __launch_bounds__(32) ctc_prefix_beam_kernel(const CtcArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  Work& w = *reinterpret_cast<Work*>(smem);
  uint32_t* allow = reinterpret_cast<uint32_t*>(smem + sizeof(Work));      // keyword-token bitmap over V (optional)
  const int lane = threadIdx.x;
  const long long b = blockIdx.x;
  const int V = a.V, SB = a.score_beam;
  long long n = a.lens ? (long long)a.lens[b] : a.T;
  n = n < 0 ? 0 : (n > a.T ? a.T : n);

  build_allow(allow, V, a.allowed, a.n_allowed, lane);
  if (lane == 0) {
    // hypotheses: carried state or the initial [(tuple(), (1.0, 0.0, []))]
    Work* st = a.state ? reinterpret_cast<Work*>(a.state + (size_t)b * sizeof(Work)) : nullptr;
    if (st && !a.reset_state) {
      w.ncur = st->ncur; w.npool = st->npool; w.overflow = st->overflow;
      for (int h = 0; h < st->ncur; ++h) w.cur[h] = st->cur[h];
      for (int i = 0; i < st->npool; ++i) { w.ntok[i] = st->ntok[i]; w.nframe[i] = st->nframe[i]; w.nprob[i] = st->nprob[i]; }
    } else {
      init_hyps(w);
      w.overflow = 0;
    }
  }
  __syncwarp();

  const float* P = a.probs + b * a.T * (long long)V;
  for (long long t = 0; t < n; ++t) {
    const float* p = P + t * V;
    // ---- probs.topk(score_beam) + the 0.05 / keyword-set filter
    int s_idx[SBM];
    float s_prob[SBM];
    const int ns = warp_topk_filter(p, V, SB, allow, lane, s_idx, s_prob);
    if (ns == 0) continue;                       // loss.py:254-255: the frame is skipped entirely
    if (lane == 0) advance(w, (int)(a.frame_offset + t * a.frame_stride), s_idx, s_prob, ns, a.path_beam);
    __syncwarp();
  }

  if (lane == 0) {
    // hyps = [(prefix, pb + pnb, nodes)]
    a.nhyp[b] = w.ncur;
    a.overflow[b] = w.overflow;
    for (int h = 0; h < a.path_beam; ++h) {
      const long long o = b * a.path_beam + h;
      if (h < w.ncur) {
        const Hyp& c = w.cur[h];
        a.hyp_len[o] = c.len;
        a.hyp_score[o] = __dadd_rn(c.pb, c.pnb);
        for (int i = 0; i < ML; ++i) {
          a.hyp_tokens[o * ML + i] = i < c.len ? c.tok[i] : -1;
          a.node_frame[o * ML + i] = i < c.nlen ? w.nframe[c.node[i]] : -1;
          a.node_prob[o * ML + i] = i < c.nlen ? w.nprob[c.node[i]] : 0.f;
        }
      } else {
        a.hyp_len[o] = -1;
        a.hyp_score[o] = 0.0;
      }
    }
    if (a.state) {
      Work* st = reinterpret_cast<Work*>(a.state + (size_t)b * sizeof(Work));
      st->ncur = w.ncur; st->npool = w.npool; st->overflow = w.overflow;
      for (int h = 0; h < w.ncur; ++h) st->cur[h] = w.cur[h];
      for (int i = 0; i < w.npool; ++i) { st->ntok[i] = w.ntok[i]; st->nframe[i] = w.nframe[i]; st->nprob[i] = w.nprob[i]; }
    }
  }
}

// score_ctc.py:201-220: first hypothesis (in beam order) containing a keyword (in keyword order)
__global__ void ctc_keyword_hit_kernel(const int32_t* __restrict__ nhyp, const int32_t* __restrict__ hyp_len,
                                       const int32_t* __restrict__ hyp_tokens, const int32_t* __restrict__ node_frame,
                                       const float* __restrict__ node_prob, long long B, int path_beam,
                                       const int32_t* __restrict__ kw_tokens, const int32_t* __restrict__ kw_off, int nkw,
                                       int32_t* __restrict__ hit, double* __restrict__ hit_score,
                                       int32_t* __restrict__ start, int32_t* __restrict__ end) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  int found = -1, st = 0, en = 0;
  double score = 1.0;
  for (int h = 0; h < nhyp[b] && found < 0; ++h) {
    const long long o = b * path_beam + h;
    const int32_t* pre = hyp_tokens + o * ML;
    for (int k = 0; k < nkw; ++k) {
      const int32_t* lab = kw_tokens + kw_off[k];
      const int nl = kw_off[k + 1] - kw_off[k];
      const int off = is_sublist(pre, hyp_len[o], lab, nl);
      if (off != -1) {
        found = k;
        st = node_frame[o * ML + off];
        en = node_frame[o * ML + off + nl - 1];
        for (int i = off; i < off + nl; ++i) score = __dmul_rn(score, (double)node_prob[o * ML + i]);
        break;
      }
    }
    if (found >= 0) score = sqrt(score);
  }
  hit[b] = found; hit_score[b] = score; start[b] = st; end[b] = en;
}

}  // namespace

size_t ctc_state_bytes() { return sizeof(Work); }

int ctc_launch(const CtcArgs& a, cudaStream_t st) {
  const size_t smem = sizeof(Work) + (size_t)((a.V + 31) / 32) * 4;
  WEKWS_REQUIRE(smem <= 227 * 1024, "ctc decode: vocabulary %d too large for the shared-memory token bitmap", a.V);
  static size_t attr_bytes[64] = {0};                  // per device: the largest dynamic size opted into so far
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_bytes[dev] < smem) {
    WEKWS_CUDA_OK(cudaFuncSetAttribute(ctc_prefix_beam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_bytes[dev] = smem;
  }
  ctc_prefix_beam_kernel<<<(unsigned)a.B, 32, smem, st>>>(a);
  return check_launch("ctc_prefix_beam_kernel");
}

int ctc_hit_launch(const int32_t* nhyp, const int32_t* hyp_len, const int32_t* hyp_tokens, const int32_t* node_frame,
                   const float* node_prob, long long B, int path_beam, const int32_t* kw_tokens, const int32_t* kw_off,
                   int nkw, int32_t* hit, double* hit_score, int32_t* start, int32_t* end, cudaStream_t st) {
  const int nt = 64;
  ctc_keyword_hit_kernel<<<(unsigned)((B + nt - 1) / nt), nt, 0, st>>>(nhyp, hyp_len, hyp_tokens, node_frame, node_prob, B,
                                                                     path_beam, kw_tokens, kw_off, nkw, hit, hit_score,
                                                                     start, end);
  return check_launch("ctc_keyword_hit_kernel");
}

}  // namespace wekws

using namespace wekws;

extern "C" int64_t wekws_ctc_state_bytes(void) { return (int64_t)ctc_state_bytes(); }

extern "C" int wekws_ctc_prefix_beam_search(const float* d_probs, const int32_t* d_lens, int64_t B, int64_t T, int V,
                                            const int32_t* d_keyword_tokens, int n_keyword_tokens, int score_beam_size,
                                            int path_beam_size, int64_t frame_offset, int frame_stride, void* d_state,
                                            int reset_state, int32_t* d_nhyp, int32_t* d_hyp_len, int32_t* d_hyp_tokens,
                                            double* d_hyp_score, int32_t* d_node_frame, float* d_node_prob,
                                            int32_t* d_overflow, void* stream) {
  WEKWS_REQUIRE(B >= 0 && T >= 0 && V >= 1 && V <= 32767, "wekws_ctc_prefix_beam_search: bad sizes (vocabulary <= 32767)");
  WEKWS_REQUIRE(score_beam_size >= 1 && score_beam_size <= WEKWS_CTC_MAX_SCORE_BEAM && score_beam_size <= V,
                "score_beam_size %d out of range (1..%d)", score_beam_size, WEKWS_CTC_MAX_SCORE_BEAM);
  WEKWS_REQUIRE(path_beam_size >= 1 && path_beam_size <= WEKWS_CTC_MAX_PATH_BEAM, "path_beam_size %d out of range (1..%d)",
                path_beam_size, WEKWS_CTC_MAX_PATH_BEAM);
  WEKWS_REQUIRE(n_keyword_tokens >= 0 && (n_keyword_tokens == 0 || d_keyword_tokens), "keyword token set is null");
  WEKWS_REQUIRE(frame_stride >= 1, "frame_stride must be >= 1");
  if (B == 0) return WEKWS_OK;
  WEKWS_REQUIRE((d_probs || T == 0) && d_nhyp && d_hyp_len && d_hyp_tokens && d_hyp_score && d_node_frame && d_node_prob &&
                    d_overflow,
                "wekws_ctc_prefix_beam_search: null argument");
  CtcArgs a;
  a.probs = d_probs; a.lens = d_lens; a.B = B; a.T = T; a.V = V;
  a.allowed = d_keyword_tokens; a.n_allowed = n_keyword_tokens;
  a.score_beam = score_beam_size; a.path_beam = path_beam_size;
  a.frame_offset = frame_offset; a.frame_stride = frame_stride;
  a.state = (uint8_t*)d_state; a.reset_state = reset_state;
  a.nhyp = d_nhyp; a.overflow = d_overflow; a.hyp_len = d_hyp_len; a.hyp_tokens = d_hyp_tokens; a.hyp_score = d_hyp_score;
  a.node_frame = d_node_frame; a.node_prob = d_node_prob;
  return ctc_launch(a, (cudaStream_t)stream);
}

extern "C" int wekws_ctc_keyword_hit(const int32_t* d_nhyp, const int32_t* d_hyp_len, const int32_t* d_hyp_tokens,
                                     const int32_t* d_node_frame, const float* d_node_prob, int64_t B, int path_beam_size,
                                     const int32_t* d_kw_tokens, const int32_t* d_kw_offsets, int num_keywords,
                                     int32_t* d_hit, double* d_hit_score, int32_t* d_start, int32_t* d_end, void* stream) {
  WEKWS_REQUIRE(B >= 0 && path_beam_size >= 1 && num_keywords >= 1, "wekws_ctc_keyword_hit: bad sizes");
  if (B == 0) return WEKWS_OK;
  WEKWS_REQUIRE(d_nhyp && d_hyp_len && d_hyp_tokens && d_node_frame && d_node_prob && d_kw_tokens && d_kw_offsets && d_hit &&
                    d_hit_score && d_start && d_end,
                "wekws_ctc_keyword_hit: null argument");
  return ctc_hit_launch(d_nhyp, d_hyp_len, d_hyp_tokens, d_node_frame, d_node_prob, B, path_beam_size, d_kw_tokens,
                        d_kw_offsets, num_keywords, d_hit, d_hit_score, d_start, d_end, (cudaStream_t)stream);
}
