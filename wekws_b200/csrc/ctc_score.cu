// Evaluation half of the CTC recipes on the device (examples/hi_xiaowen/s0/run_ctc.sh stage 3):
//   ctc_stream_score_kernel  wekws/bin/stream_score_ctc.py:209-381 -- per utterance the per-frame beam step
//                            (ctc_beam.cuh, the same step as stream_kws_ctc.py:124-215) and the script's own detection
//   ctc_det_sweep_kernel     wekws/bin/compute_det_ctc.py:251-281 -- false rejects / false alarms per threshold
// The label / score-file join of compute_det_ctc.py:50-124 is string work and stays on the host
// (wekws_b200/ctc_score.py).
//
// The detection of stream_score_ctc.py differs from execute_detection in stream_kws_ctc.py (kws_stream.cu):
//   * hit_keyword / start / end are set once per utterance, not per frame.  Once a keyword was hit and not activated,
//     the hypothesis loop stops after hyps[0] whether or not it holds a keyword, and hit_score = sqrt(hit_score) runs
//     on every such frame (:324-342); the duration gate then reads whatever start / end hold, stale or not;
//   * a frame the top-k + 0.05 + token-set filter empties is skipped entirely, detection included (:260-261);
//   * the gates are the threshold and min_frames <= end - start <= max_frames only (:345-347);
//   * an activation resets the beam, hit_keyword and hit_score (start / end keep their values) and decoding goes on to
//     the end of the utterance, so one utterance can be detected several times (:348-360).
#include <math.h>

#include "common.cuh"
#include "ctc_beam.cuh"

namespace wekws {
namespace {

using namespace beam;

struct ScoreArgs {
  const float* probs;           // (B, T, V)
  const int32_t* lens;          // (B) or null = T
  long long B, T;
  int V;
  const int32_t* allowed;       // keywords_idxset
  int n_allowed;
  const int32_t* kw_tokens;     // keyword k = kw_tokens[kw_off[k] .. kw_off[k+1])
  const int32_t* kw_off;
  int nkw;
  wekws_ctc_score_config cfg;
  int32_t* count;               // (B)
  int32_t* overflow;            // (B)
  int32_t* kw;                  // (B, max_detections)
  double* score;
  int32_t* start;
  int32_t* end;
};

__global__ void __launch_bounds__(32) ctc_stream_score_kernel(const ScoreArgs a) {
  extern __shared__ __align__(16) uint8_t smem[];
  Work& w = *reinterpret_cast<Work*>(smem);
  uint32_t* allow = reinterpret_cast<uint32_t*>(smem + sizeof(Work));
  const int lane = threadIdx.x;
  const long long b = blockIdx.x;
  long long n = a.lens ? (long long)a.lens[b] : a.T;
  n = n < 0 ? 0 : (n > a.T ? a.T : n);

  build_allow(allow, a.V, a.allowed, a.n_allowed, lane);
  if (lane == 0) {                               // :228
    init_hyps(w);
    w.overflow = 0;
  }
  __syncwarp();

  // :230-234, once per utterance
  int hit = -1, start = 0, end = 0, count = 0;
  double hit_score = 1.0;
  const int maxdet = a.cfg.max_detections;
  const float* P = a.probs + b * a.T * (long long)a.V;
  for (long long t = 0; t < n; ++t) {
    int s_idx[SBM];
    float s_prob[SBM];
    const int ns = warp_topk_filter(P + t * a.V, a.V, a.cfg.score_beam, allow, lane, s_idx, s_prob);
    if (ns == 0) continue;                       // :260-261: no beam change and no detection on this frame
    if (lane == 0) {
      advance(w, (int)(t * a.cfg.frame_skip), s_idx, s_prob, ns, a.cfg.path_beam);
      // :324-342.  With hit >= 0 carried from an earlier frame the loop ends after hyps[0] in any case.
      for (int h = 0; h < w.ncur; ++h) {
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
        if (hit >= 0) {
          hit_score = sqrt(hit_score);
          break;
        }
      }
      const int duration = end - start;          // :344-360
      if (hit >= 0 && hit_score >= a.cfg.threshold && a.cfg.min_frames <= duration && duration <= a.cfg.max_frames) {
        if (count < maxdet) {
          const long long o = b * maxdet + count;
          a.kw[o] = hit; a.score[o] = hit_score; a.start[o] = start; a.end[o] = end;
        }
        ++count;
        init_hyps(w);
        hit = -1;
        hit_score = 1.0;
      }
    }
    __syncwarp();
  }
  if (lane == 0) {
    a.count[b] = count;
    a.overflow[b] = w.overflow;
  }
}

// One block per threshold: false rejects #(kw < thr) and false alarms #(filler >= thr), compared in double
__global__ void __launch_bounds__(256) ctc_det_sweep_kernel(const double* __restrict__ kw, long long n_kw,
                                                            const double* __restrict__ filler, long long n_filler,
                                                            const double* __restrict__ thr,
                                                            long long* __restrict__ false_reject,
                                                            long long* __restrict__ false_alarm) {
  __shared__ long long part[2][8];
  const double th = thr[blockIdx.x];
  long long fr = 0, fa = 0;
  for (long long i = threadIdx.x; i < n_kw; i += blockDim.x) fr += __ldg(kw + i) < th;
  for (long long i = threadIdx.x; i < n_filler; i += blockDim.x) fa += __ldg(filler + i) >= th;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    fr += __shfl_xor_sync(0xffffffffu, fr, o);
    fa += __shfl_xor_sync(0xffffffffu, fa, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { part[0][warp] = fr; part[1][warp] = fa; }
  __syncthreads();
  if (threadIdx.x == 0) {
    fr = 0; fa = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { fr += part[0][i]; fa += part[1][i]; }
    false_reject[blockIdx.x] = fr;
    false_alarm[blockIdx.x] = fa;
  }
}

}  // namespace
}  // namespace wekws

using namespace wekws;

extern "C" int wekws_ctc_stream_score(const float* d_probs, const int32_t* d_lens, int64_t B, int64_t T, int V,
                                      const int32_t* d_token_set, int n_tokens, const int32_t* d_kw_tokens,
                                      const int32_t* d_kw_offsets, int num_keywords, const wekws_ctc_score_config* cfg,
                                      int32_t* d_count, int32_t* d_overflow, int32_t* d_kw, double* d_score,
                                      int32_t* d_start, int32_t* d_end, void* stream) {
  WEKWS_REQUIRE(cfg, "wekws_ctc_stream_score: null config");
  WEKWS_REQUIRE(B >= 0 && T >= 0 && V >= 1 && V <= 32767, "wekws_ctc_stream_score: bad sizes (vocabulary <= 32767)");
  WEKWS_REQUIRE(cfg->score_beam >= 1 && cfg->score_beam <= WEKWS_CTC_MAX_SCORE_BEAM && cfg->score_beam <= V,
                "score_beam %d out of range (1..%d)", cfg->score_beam, WEKWS_CTC_MAX_SCORE_BEAM);
  WEKWS_REQUIRE(cfg->path_beam >= 1 && cfg->path_beam <= WEKWS_CTC_MAX_PATH_BEAM, "path_beam %d out of range (1..%d)",
                cfg->path_beam, WEKWS_CTC_MAX_PATH_BEAM);
  WEKWS_REQUIRE(cfg->frame_skip >= 1, "frame_skip must be >= 1");
  WEKWS_REQUIRE(cfg->max_detections >= 1, "max_detections must be >= 1");
  WEKWS_REQUIRE(T * (int64_t)cfg->frame_skip < (1ll << 31), "wekws_ctc_stream_score: T * frame_skip exceeds int32 frames");
  WEKWS_REQUIRE(num_keywords >= 1 && n_tokens >= 0, "wekws_ctc_stream_score: at least one keyword is needed");
  if (B == 0) return WEKWS_OK;
  WEKWS_REQUIRE((d_probs || T == 0) && d_kw_tokens && d_kw_offsets && d_count && d_overflow && d_kw && d_score &&
                    d_start && d_end && (n_tokens == 0 || d_token_set),
                "wekws_ctc_stream_score: null argument");
  WEKWS_REQUIRE(B < (1ll << 31), "wekws_ctc_stream_score: too many utterances");
  ScoreArgs a;
  a.probs = d_probs; a.lens = d_lens; a.B = B; a.T = T; a.V = V;
  a.allowed = d_token_set; a.n_allowed = n_tokens;
  a.kw_tokens = d_kw_tokens; a.kw_off = d_kw_offsets; a.nkw = num_keywords;
  a.cfg = *cfg;
  a.count = d_count; a.overflow = d_overflow; a.kw = d_kw; a.score = d_score; a.start = d_start; a.end = d_end;
  const size_t smem = sizeof(Work) + (size_t)((V + 31) / 32) * 4;
  WEKWS_REQUIRE(smem <= 227 * 1024, "ctc stream score: vocabulary %d too large for the shared-memory token bitmap", V);
  static size_t attr_bytes[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && attr_bytes[dev] < smem) {
    WEKWS_CUDA_OK(cudaFuncSetAttribute(ctc_stream_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_bytes[dev] = smem;
  }
  ctc_stream_score_kernel<<<(unsigned)B, 32, smem, (cudaStream_t)stream>>>(a);
  return check_launch("ctc_stream_score_kernel");
}

extern "C" int wekws_ctc_det_sweep(const double* d_conf_kw, int64_t n_kw, const double* d_conf_filler,
                                   int64_t n_filler, const double* d_thresholds, int nthr, int64_t* d_false_reject,
                                   int64_t* d_false_alarm, void* stream) {
  WEKWS_REQUIRE(n_kw >= 0 && n_filler >= 0 && nthr >= 0, "wekws_ctc_det_sweep: bad sizes");
  if (nthr == 0) return WEKWS_OK;
  WEKWS_REQUIRE((d_conf_kw || n_kw == 0) && (d_conf_filler || n_filler == 0) && d_thresholds && d_false_reject &&
                    d_false_alarm,
                "wekws_ctc_det_sweep: null argument");
  ctc_det_sweep_kernel<<<(unsigned)nthr, 256, 0, (cudaStream_t)stream>>>(d_conf_kw, n_kw, d_conf_filler, n_filler,
                                                                         d_thresholds, (long long*)d_false_reject,
                                                                         (long long*)d_false_alarm);
  return check_launch("ctc_det_sweep_kernel");
}
