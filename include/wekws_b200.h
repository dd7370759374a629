/*
 * wekws_b200 -- C ABI of the B200-native WeKws streaming keyword-spotting forward path.
 *
 * Plain C, no torch / ATen / C++ types cross this boundary.  Every pointer named
 * d_* is a device pointer on the CURRENT CUDA device; h_* is a host pointer.
 * `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 * Every function returns 0 on success and a negative wekws_status on failure;
 * wekws_last_error() then holds a thread-local human-readable message.  Nothing
 * throws, nothing allocates device memory inside a *_forward call except a
 * per-handle scratch buffer that grows monotonically on first use.
 *
 * What each entry point replaces in the reference (wenet-e2e/wekws @ 1a8ee65):
 *
 *   wekws_fbank_*          torchaudio.compliance.kaldi.fbank as called by
 *                          wekws/dataset/processor.py:173-203 (compute_fbank) and
 *                          wekws/bin/stream_kws_ctc.py:335-364 (accept_wave), fused with
 *                          GlobalCMVN.forward wekws/model/cmvn.py:37-48; native twin:
 *                          wenet::Fbank::Compute runtime/core/frontend/fbank.h:138-198
 *                          behind FeaturePipeline::AcceptWaveform
 *                          runtime/core/frontend/feature_pipeline.cc:30-47.
 *   wekws_model_create /   init_model(configs) wekws/model/kws_model.py:97-214 followed by
 *   _set_tensor/_finalize  load_checkpoint -> load_state_dict wekws/utils/checkpoint.py:23-36;
 *                          tensor names ARE the reference state_dict keys (SURVEY.md 8b).
 *   wekws_model_forward    KWSModel.forward(x, in_cache) wekws/model/kws_model.py:65-76
 *                          (and forward_softmax :78-90 via WEKWS_ACT_SIGMOID/IDENTITY +
 *                          WEKWS_FWD_SOFTMAX); native twin: KeywordSpotting::Forward
 *                          runtime/core/kws/keyword_spotting.cc:56-95 whose ONNX graph has
 *                          inputs (input, cache) and outputs (output, r_cache).
 *   wekws_pipeline_forward the composition the callers perform: Fbank -> model, i.e.
 *                          stream_kws_ctc.py:482-487 / score.py:117-127, raw PCM in,
 *                          posteriors out.
 *   wekws_kws_*            the streaming CTC keyword spotter around them: KeyWordSpotter
 *                          wekws/bin/stream_kws_ctc.py:218-529 (PCM / feature carries,
 *                          per-frame beam step + execute_detection, reset / reset_all).
 *   wekws_ctc_stream_score the test-set scorer wekws/bin/stream_score_ctc.py:209-381 (per
 *                          utterance: per-frame beam step + the script's own detection).
 *   wekws_ctc_det_sweep    the threshold sweep of wekws/bin/compute_det_ctc.py:251-281.
 */
#ifndef WEKWS_B200_H_
#define WEKWS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WEKWS_B200_ABI_VERSION 6   /* 2: + wekws_fbank_set_mfcc, wekws_fbank_feature_dim, wekws_det_stats; 3: det max_score is double; 4: precision mode 2, wekws_model_uses_tensor_cores_bt; 5: + wekws_kws_* streaming keyword spotter; 6: + wekws_ctc_stream_score, wekws_ctc_det_sweep */

#if defined(__GNUC__)
#define WEKWS_API __attribute__((visibility("default")))
#else
#define WEKWS_API
#endif

typedef enum {
  WEKWS_OK = 0,
  WEKWS_ERR_INVALID = -1,     /* bad argument / unsupported configuration              */
  WEKWS_ERR_CUDA = -2,        /* a CUDA runtime call failed (message has the string)  */
  WEKWS_ERR_STATE = -3,       /* call order: forward before finalize, missing tensor  */
  WEKWS_ERR_NOMEM = -4
} wekws_status;

typedef enum {
  WEKWS_BACKBONE_MDTC = 0,    /* wekws/model/mdtc.py  MDTC                             */
  WEKWS_BACKBONE_TCN = 1,     /* wekws/model/tcn.py   TCN(block_class=CnnBlock)        */
  WEKWS_BACKBONE_DSTCN = 2,   /* wekws/model/tcn.py   TCN(block_class=DsCnnBlock)      */
  WEKWS_BACKBONE_GRU = 3,     /* torch.nn.GRU, kws_model.py:128-133                    */
  WEKWS_BACKBONE_FSMN = 4     /* wekws/model/fsmn.py FSMN (preprocessing none, classifier identity,
                                 kws_model.py:158-170,121-122,191): tensors backbone.in_linear{1,2}.linear.*,
                                 backbone.fsmn.{l}.{0.linear.weight,1.conv_left.weight,1.conv_right.weight,
                                 2.linear.*}, backbone.out_linear{1,2}.linear.*                    */
} wekws_backbone;

typedef enum { WEKWS_ACT_IDENTITY = 0, WEKWS_ACT_SIGMOID = 1 } wekws_activation;
typedef enum { WEKWS_PCM_S16 = 0, WEKWS_PCM_F32 = 1 } wekws_pcm_dtype;
typedef enum { WEKWS_WINDOW_POVEY = 0, WEKWS_WINDOW_HAMMING = 1 } wekws_window;

/* forward flags */
#define WEKWS_FWD_SOFTMAX 1u  /* apply softmax over odim after the activation (forward_softmax) */

WEKWS_API const char* wekws_last_error(void);
WEKWS_API int wekws_abi_version(void);
/* Number of kernels this library has launched since load (all handles, all threads). */
WEKWS_API uint64_t wekws_launch_count(void);

/* ----------------------------------------------------------------------------- Fbank */
typedef struct wekws_fbank wekws_fbank;

typedef struct {
  int32_t sample_rate;     /* 16000                                                   */
  int32_t frame_length;    /* samples per frame, 400  (frame_length=25 ms)            */
  int32_t frame_shift;     /* samples per hop,   160  (frame_shift=10 ms)             */
  int32_t n_fft;           /* 512 (round_to_power_of_two); only 512 is implemented    */
  int32_t num_mel_bins;    /* <= 128                                                  */
  float   preemphasis;     /* 0.97                                                    */
  int32_t remove_dc;       /* 1                                                       */
  float   log_floor;       /* FLT_EPSILON (kaldi.py:21)                               */
} wekws_fbank_config;

/* h_window: frame_length floats (Povey / Hamming, computed by the host exactly as
 * kaldi.py:88-110 does).  h_mel: num_mel_bins x (n_fft/2) row-major mel weights
 * (kaldi.py:436-511; the Nyquist column is implicitly zero, kaldi.py:627).        */
WEKWS_API int wekws_fbank_create(const wekws_fbank_config* cfg, const float* h_window,
                       const float* h_mel, wekws_fbank** out);
WEKWS_API void wekws_fbank_destroy(wekws_fbank* fb);
/* Frames produced for num_samples samples (snip_edges=True): 0 if < frame_length.   */
WEKWS_API int64_t wekws_fbank_num_frames(const wekws_fbank* fb, int64_t num_samples);
WEKWS_API int wekws_fbank_num_mel_bins(const wekws_fbank* fb);

/* MFCC mode (SURVEY 8f-1): the front-end of the shipped mdtc / mdtc_small configs
 * (examples/hi_xiaowen/s0/conf/mdtc.yaml:8-14 `feature_type: mfcc`), i.e.
 * torchaudio.compliance.kaldi.mfcc as called by wekws/dataset/processor.py:157-166 (compute_mfcc):
 * the log-mel row times a DCT-II matrix h_dct[num_mel_bins][num_ceps] (ortho, first column sqrt(1/num_mel_bins)),
 * times h_lifter[num_ceps] (NULL = no liftering), then the optional CMVN of wekws_fbank_forward over the
 * num_ceps outputs.  After this call wekws_fbank_forward writes (B, max_frames, num_ceps).  num_ceps = 0
 * switches back to log-mel output.  wekws_fbank_feature_dim = row width of the output in the current mode. */
WEKWS_API int wekws_fbank_set_mfcc(wekws_fbank* fb, int num_ceps, const float* h_dct, const float* h_lifter);
WEKWS_API int wekws_fbank_feature_dim(const wekws_fbank* fb);

/* d_pcm: B waveforms, row b at d_pcm + b*pcm_stride elements, int16-scale values.
 * d_lens: optional per-waveform sample counts (NULL = all num_samples).
 * d_mean/d_istd: optional CMVN (NULL, NULL = none; istd NULL = mean only).
 * d_out: (B, max_frames, num_mel_bins) fp32; rows past a waveform's frame count are
 * zero-filled.  max_frames must be >= wekws_fbank_num_frames(num_samples).          */
WEKWS_API int wekws_fbank_forward(wekws_fbank* fb, const void* d_pcm, int pcm_dtype, int64_t B,
                        int64_t num_samples, int64_t pcm_stride, const int32_t* d_lens,
                        const float* d_mean, const float* d_istd, float* d_out,
                        int64_t max_frames, void* stream);

/* ----------------------------------------------------------------------------- model */
typedef struct wekws_model wekws_model;

typedef struct {
  int32_t backbone;        /* wekws_backbone                                           */
  int32_t idim;            /* input_dim  (<= 128)                                      */
  int32_t hdim;            /* hidden_dim: 32/64/128/256 for conv backbones, 128 GRU    */
  int32_t odim;            /* output_dim                                               */
  int32_t num_layers;      /* TCN/DSTCN blocks or GRU layers; MDTC: ignored            */
  int32_t num_stack;       /* MDTC only                                                */
  int32_t stack_size;      /* MDTC only                                                */
  int32_t kernel_size;     /* conv taps (mdtc 5, tcn 8)                                */
  int32_t activation;      /* wekws_activation                                         */
  int32_t norm_var;        /* cmvn.norm_var; used when global_cmvn.* tensors are set   */
  /* FSMN only (fsmn_ctc.yaml:40-52); num_layers = FSMN layers; the memory blocks always use strides 1,1 as the
   * reference builds them (fsmn.py:384-391); cache (B, proj_dim, left_order - 1 + right_order, num_layers)  */
  int32_t fsmn_input_affine_dim, fsmn_linear_dim, fsmn_proj_dim;
  int32_t fsmn_left_order, fsmn_right_order, fsmn_output_affine_dim;
} wekws_model_config;

WEKWS_API int wekws_model_create(const wekws_model_config* cfg, wekws_model** out);
WEKWS_API void wekws_model_destroy(wekws_model* m);
/* Total cache columns == backbone.padding (mdtc 244, tcn/ds_tcn 105; FSMN lorder-1+rorder); 0 for GRU. */
WEKWS_API int wekws_model_padding(const wekws_model* m);
/* name: reference state_dict key, e.g. "backbone.blocks.0.res_blocks.1.bn1.running_var".
 * Data is copied.  num_batches_tracked entries may be skipped.                      */
WEKWS_API int wekws_model_set_tensor(wekws_model* m, const char* name, const float* h_data, int64_t numel);
/* Host half of finalize: folds every eval-mode BatchNorm into its producer and packs the
 * weight stream.  No CUDA call -- usable (and tested) on a machine without a GPU.        */
WEKWS_API int wekws_model_pack(wekws_model* m);
/* wekws_model_pack + upload to the current device.                                       */
WEKWS_API int wekws_model_finalize(wekws_model* m);
/* Arithmetic of the dense GEMMs: 0 = auto (default): tcgen05 tensor cores with a 3-pass bf16
 * operand split (~2^-17 relative, posteriors within 1e-5 of fp32) where a fused tensor-core
 * kernel exists (mdtc / dense tcn with hidden 64, ds_tcn with hidden 256 and k = 8; chunk >= 8 frames),
 * FP32 FMA elsewhere; the GRU (hidden 128, 1-2 layers) has a weight-streaming tcgen05 kernel that auto picks by batch
 * and chunk (>= 640 streams at T = 1, >= 400 at T = 2..7, >= 256 at T >= 8) and the FP32 kernel otherwise; 1 = FP32 FMA only;
 * 2 = the tensor-core kernel wherever one exists, whatever the batch (tests, benchmarks). */
WEKWS_API int wekws_model_set_precision(wekws_model* m, int mode);
/* 1 if a forward with T frames per call runs the tcgen05 kernel (after finalize), else 0.  The plain form answers for
 * a large batch; the GRU's choice also depends on the batch B.                               */
WEKWS_API int wekws_model_uses_tensor_cores(const wekws_model* m, int64_t T);
WEKWS_API int wekws_model_uses_tensor_cores_bt(const wekws_model* m, int64_t B, int64_t T);
/* Debug/test accessors of the packed host-side program (valid after finalize).      */
WEKWS_API int64_t wekws_model_packed_floats(const wekws_model* m, int which /*0 stream, 1 vectors, 2 tensor-core weight images (bytes / 4), 3 tensor-core classifier images (bytes / 4)*/);
WEKWS_API int wekws_model_packed_copy(const wekws_model* m, int which, float* h_dst, int64_t capacity);

/* d_feats (B,T,idim); d_in_cache NULL (start of stream == zeros) or
 * conv: (B,hdim,padding)  GRU: (num_layers,B,hdim)  FSMN: (B,proj_dim,padding,num_layers); d_out (B,T,odim);
 * d_out_cache same shape as the cache; it may be the SAME buffer as d_in_cache (in-place
 * streaming update: every slice is read before it is overwritten) or a disjoint one, not a
 * partially overlapping one.                                                       */
WEKWS_API int wekws_model_forward(wekws_model* m, const float* d_feats, const float* d_in_cache,
                        float* d_out, float* d_out_cache, int64_t B, int64_t T,
                        uint32_t flags, void* stream);

/* Detection statistics of max-pooling keyword models on the device (SURVEY 8f-2), bit-exact with the host
 * pipeline wekws/bin/score.py:128-137 ('{:.6f}' score file) -> wekws/bin/compute_det.py:76-105:
 *   d_max_score[b,k]   = max over the first lens[b] frames of the text-rounded posterior as the DOUBLE Python parses
 *                        back from the score file (false-reject test `max < threshold` is done in double),
 *   d_triggers[b,k,i]  = triggers of the left-to-right scan "score >= thresholds[i] -> count, skip window_shift
 *                        frames" (false alarms).
 * d_post (B,T,K) posteriors; d_lens NULL = all T frames; d_thresholds nthr doubles (the host accumulates
 * threshold += step exactly as the reference does).                                                   */
WEKWS_API int wekws_det_stats(const float* d_post, const int32_t* d_lens, int64_t B, int64_t T, int K,
                    const double* d_thresholds, int nthr, int window_shift, double* d_max_score,
                    int32_t* d_triggers, void* stream);

/* CTC prefix beam search + keyword look-up on the device (SURVEY 8f-2, CTC models), bit-exact with the reference's pure
 * Python: wekws/model/loss.py:206-312 ctc_prefix_beam_search as called by wekws/bin/score_ctc.py:198-200 (whole
 * utterance) and its per-frame streaming twin wekws/bin/stream_kws_ctc.py:124-215,400-409 (hypotheses carried in
 * d_state between calls; frame numbers = frame_offset + row * frame_stride), then the look-up of
 * score_ctc.py:201-220 / stream_kws_ctc.py:411-434.
 *   d_probs (B,T,V) softmax posteriors; d_lens NULL = T frames; d_keyword_tokens: the keywords' token-id set
 *   (n = 0: no filter); d_state: B x wekws_ctc_state_bytes() bytes or NULL (reset_state != 0: start from the empty
 *   hypothesis and write the final state).
 * Outputs per utterance, hypotheses in beam order: d_nhyp (B); d_hyp_len (B,path_beam) (-1 = unused);
 *   d_hyp_tokens / d_node_frame / d_node_prob (B,path_beam,WEKWS_CTC_MAX_PREFIX); d_hyp_score (B,path_beam) = pb + pnb
 *   (double, as Python computes it); d_overflow (B) != 0 if a prefix outgrew WEKWS_CTC_MAX_PREFIX tokens.          */
#define WEKWS_CTC_MAX_PREFIX 64
#define WEKWS_CTC_MAX_PATH_BEAM 20
#define WEKWS_CTC_MAX_SCORE_BEAM 3
WEKWS_API int64_t wekws_ctc_state_bytes(void);
WEKWS_API int wekws_ctc_prefix_beam_search(const float* d_probs, const int32_t* d_lens, int64_t B, int64_t T, int V,
                                 const int32_t* d_keyword_tokens, int n_keyword_tokens, int score_beam_size,
                                 int path_beam_size, int64_t frame_offset, int frame_stride, void* d_state,
                                 int reset_state, int32_t* d_nhyp, int32_t* d_hyp_len, int32_t* d_hyp_tokens,
                                 double* d_hyp_score, int32_t* d_node_frame, float* d_node_prob, int32_t* d_overflow,
                                 void* stream);
/* d_kw_tokens: the keywords' token sequences back to back, keyword k = [d_kw_offsets[k], d_kw_offsets[k+1]).
 * d_hit (B) = index of the detected keyword or -1; d_hit_score = sqrt(product of its token probabilities);
 * d_start / d_end = frames of its first / last token.                                                        */
WEKWS_API int wekws_ctc_keyword_hit(const int32_t* d_nhyp, const int32_t* d_hyp_len, const int32_t* d_hyp_tokens,
                          const int32_t* d_node_frame, const float* d_node_prob, int64_t B, int path_beam_size,
                          const int32_t* d_kw_tokens, const int32_t* d_kw_offsets, int num_keywords, int32_t* d_hit,
                          double* d_hit_score, int32_t* d_start, int32_t* d_end, void* stream);

/* Context expansion + frame skipping of the FSMN / CTC recipes (SURVEY 8f-4): wekws/dataset/processor.py:267-312
 * (batched twin wekws/dataset/init_dataset.py:24-68).  d_feats (B,T,D); d_lens NULL = all T frames valid;
 * d_out (B, out_frames, D*(left+right+1)): row i of stream b = concat(feats[max(i*skip+k-left, 0)], k = 0..left+right)
 * for i < wekws_context_expand_frames(lens[b], right, skip), zeros after.                                      */
WEKWS_API int64_t wekws_context_expand_frames(int64_t num_frames, int right, int skip);
WEKWS_API int wekws_context_expand(const float* d_feats, const int32_t* d_lens, int64_t B, int64_t T, int D, int left,
                         int right, int skip, float* d_out, int64_t out_frames, void* stream);

/* ------------------------------------------------------------------ streaming CTC keyword spotter
 * KeyWordSpotter of wekws/bin/stream_kws_ctc.py:218-529 for B streams at once, bit-exact (wekws_b200/spotter.py drives
 * it).  The host plans every row count and offset from the sample counts it knows; nothing here is read back to plan.
 *
 * wekws_kws_splice  accept_wave :346-364: stage[b] = carry_in[b][0..carry_len) ++ pcm[b][0..new_len) (int16, row
 *   stride stage_stride, for wekws_fbank_forward with d_lens = carry_len + new_len), and carry_out[b] = stage[b] from
 *   sample consumed[b] on (the samples the Fbank frames did not use).  carry_in / carry_out: (B, carry_cap), distinct.
 * wekws_kws_context accept_wave :366-397: d_feats (B,T,D) Fbank rows, d_num_frames (B) rows per stream.  With expand,
 *   the rows are context-expanded with the carried rows d_carry_in (B, left+right, D), d_carry_len (B) rows (-1 =
 *   first chunk: left copies of row 0), and the next carry is written to d_carry_out (the last min(left+right, nf) rows;
 *   the old carry when nf == 0).  Then every skip-th row from d_skip_offset[b] on is written to d_out at packed row
 *   d_row_offsets[b], d_rows[b] rows (width D*(left+right+1) with expand, D without); max_rows = max of d_rows.
 * wekws_kws_detect  forward :489-512: per stream d_rows[b] rows of softmax posteriors at d_probs + d_row_offsets[b]*V,
 *   each one streaming beam step (wekws_ctc_prefix_beam_search's) then execute_detection :411-480; after an activation
 *   the beam is reset and the rest of the chunk is skipped; at the end of the chunk a top hypothesis whose first token
 *   is more than max_frames old is reset.  d_token_set: keywords_idxset; d_kw_tokens / d_kw_offsets as in
 *   wekws_ctc_keyword_hit, in dict order.  d_state: B x wekws_kws_state_bytes(), set up by wekws_kws_reset(full = 1).
 *   d_result (B, WEKWS_KWS_RESULT_FIELDS) int64: state (-1 = no rows: the reference returns {}, 0, 1 = activated),
 *   keyword index (-1), start frame, end frame, score (the bits of the double hit_score), overflow (a prefix outgrew
 *   WEKWS_CTC_MAX_PREFIX tokens or the node pool filled since the last full reset; the results are then not exact).
 * wekws_kws_reset   reset() :516-519 (full = 0) or the decoder part of reset_all() :521-529 (full = 1: also
 *   total_frames, last_active_pos, the overflow flag) of the listed streams (d_streams NULL: streams 0..B-1).       */
#define WEKWS_KWS_RESULT_FIELDS 6
typedef struct {
  double threshold;          /* activation: hit_score >= threshold                                           */
  int32_t min_frames;        /* and min_frames <= end - start <= max_frames                                  */
  int32_t max_frames;
  int32_t interval_frames;   /* and (no activation yet or end - last_active_pos >= interval_frames)          */
  int32_t score_beam;        /* 1..WEKWS_CTC_MAX_SCORE_BEAM                                                  */
  int32_t path_beam;         /* 1..WEKWS_CTC_MAX_PATH_BEAM                                                   */
  int32_t frame_skip;        /* row t of a chunk is frame total_frames + t * frame_skip                      */
} wekws_kws_config;

WEKWS_API int64_t wekws_kws_state_bytes(void);
WEKWS_API int wekws_kws_reset(void* d_state, int64_t B, const int32_t* d_streams, int64_t n_streams, int full,
                              void* stream);
WEKWS_API int wekws_kws_detect(const float* d_probs, const int32_t* d_row_offsets, const int32_t* d_rows, int64_t B,
                               int V, const int32_t* d_token_set, int n_tokens, const int32_t* d_kw_tokens,
                               const int32_t* d_kw_offsets, int num_keywords, const wekws_kws_config* cfg,
                               void* d_state, int64_t* d_result, void* stream);
WEKWS_API int wekws_kws_splice(const int16_t* d_pcm, int64_t pcm_stride, const int32_t* d_new_len,
                               const int32_t* d_carry_len, const int32_t* d_consumed, const int16_t* d_carry_in,
                               int16_t* d_carry_out, int64_t carry_cap, int16_t* d_stage, int64_t stage_stride,
                               int64_t B, void* stream);
WEKWS_API int wekws_kws_context(const float* d_feats, int64_t B, int64_t T, int D, const int32_t* d_num_frames,
                                const float* d_carry_in, const int32_t* d_carry_len, float* d_carry_out, int left,
                                int right, int expand, int skip, const int32_t* d_skip_offset,
                                const int32_t* d_row_offsets, const int32_t* d_rows, int64_t max_rows, float* d_out,
                                void* stream);

/* ------------------------------------------------------------------ CTC test-set scoring and DET statistics
 * wekws_ctc_stream_score  wekws/bin/stream_score_ctc.py:209-381 for B utterances, bit-exact: d_probs (B,T,V) softmax
 *   posteriors, d_lens (B) valid rows (NULL = T; values outside [0, T] are clamped), row t is frame t * frame_skip.
 *   d_token_set: keywords_idxset (n_tokens = 0: no filter); d_kw_tokens / d_kw_offsets as in wekws_ctc_keyword_hit,
 *   in dict order.  Per utterance: d_count (B) activations (always exact), d_overflow (B) != 0 if a prefix outgrew
 *   WEKWS_CTC_MAX_PREFIX tokens or the node pool filled (the results are then not exact), and the first
 *   min(count, max_detections) activations in frame order in d_kw / d_score (double hit_score) / d_start / d_end,
 *   each (B, max_detections).
 * wekws_ctc_det_sweep  compute_det_ctc.py:251-281 for one keyword: d_false_reject[i] = #(d_conf_kw < thr[i]),
 *   d_false_alarm[i] = #(d_conf_filler >= thr[i]), compared in double; d_thresholds as the host accumulates them. */
typedef struct {
  double threshold;          /* activation: hit_score >= threshold                                           */
  int32_t min_frames;        /* and min_frames <= end - start <= max_frames                                  */
  int32_t max_frames;
  int32_t score_beam;        /* 1..WEKWS_CTC_MAX_SCORE_BEAM                                                  */
  int32_t path_beam;         /* 1..WEKWS_CTC_MAX_PATH_BEAM                                                   */
  int32_t frame_skip;        /* dataset_conf.frame_skip: row t is frame t * frame_skip                       */
  int32_t max_detections;    /* >= 1: detections stored per utterance                                        */
} wekws_ctc_score_config;

WEKWS_API int wekws_ctc_stream_score(const float* d_probs, const int32_t* d_lens, int64_t B, int64_t T, int V,
                                     const int32_t* d_token_set, int n_tokens, const int32_t* d_kw_tokens,
                                     const int32_t* d_kw_offsets, int num_keywords, const wekws_ctc_score_config* cfg,
                                     int32_t* d_count, int32_t* d_overflow, int32_t* d_kw, double* d_score,
                                     int32_t* d_start, int32_t* d_end, void* stream);
WEKWS_API int wekws_ctc_det_sweep(const double* d_conf_kw, int64_t n_kw, const double* d_conf_filler, int64_t n_filler,
                                  const double* d_thresholds, int nthr, int64_t* d_false_reject,
                                  int64_t* d_false_alarm, void* stream);

/* Raw PCM -> posteriors: Fbank(+CMVN from the model's global_cmvn.* if set) -> model.
 * d_feat_scratch: (B, frames, idim) floats of workspace owned by the caller.        */
WEKWS_API int wekws_pipeline_forward(wekws_fbank* fb, wekws_model* m, const void* d_pcm, int pcm_dtype,
                           int64_t B, int64_t num_samples, int64_t pcm_stride,
                           float* d_feat_scratch, const float* d_in_cache, float* d_out,
                           float* d_out_cache, uint32_t flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* WEKWS_B200_H_ */
