"""CPU oracle of the streaming CTC keyword spotter: one stream of wekws/bin/stream_kws_ctc.py KeyWordSpotter.

TEST INFRASTRUCTURE ONLY (like kws_oracle.py, whose fbank, ctc_prefix_beam_search and is_sublist it reuses).  It
restates, statement for statement, what the reference's class does for one stream (line numbers of
wekws/bin/stream_kws_ctc.py):

* accept_wave    :335-398  PCM carry, kaldi fbank, context expansion with carried rows, frame skip with carried offset
* forward        :482-514  model + softmax(2), per row one beam step and execute_detection, stop after an
                           activation, total_frames, the max_frames reset
* execute_detection :411-480, reset :516-519, reset_all :521-529

Pinned by tests/golden/kws_stream.npz, which oracle/make_kws_stream_golden.py makes by running the reference class.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

from . import kws_oracle as O


class KeyWordSpotter:
    """model_fn(feats (1, T, D) float32, cache) -> (logits (1, T, V), cache); None = feed probabilities through
    forward_probs() instead.  fbank_fn(wave (N,) float32) -> (m, num_mel_bins): the Kaldi fbank (default: the oracle's
    restatement; tests pass the device Fbank to check the data movement after it bit for bit)."""

    def __init__(self, keywords_token, threshold, model_fn=None, num_mel_bins=80, frame_length=25, frame_shift=10,
                 context=None, frame_skip=1, min_frames=5, max_frames=250, interval_frames=50, score_beam=3,
                 path_beam=20, fbank_fn=None):
        self.sample_rate = 16000
        self.fbank_fn = fbank_fn
        self.num_mel_bins, self.frame_length, self.frame_shift = num_mel_bins, frame_length, frame_shift
        self.downsampling = frame_skip                                                   # :250
        self.resolution = self.frame_shift / 1000                                        # :251
        self.context_expansion = context is not None                                     # :253-259
        self.left_context, self.right_context = context if context is not None else (0, 0)
        self.model_fn = model_fn
        self.score_beam, self.path_beam = score_beam, path_beam
        self.threshold, self.min_frames, self.max_frames = threshold, min_frames, max_frames
        self.interval_frames = interval_frames
        self.keywords_token = keywords_token                                             # set_keywords :304-333
        self.keywords_idxset = {0}
        for w in keywords_token:
            self.keywords_idxset.update(keywords_token[w]["token_id"])
        self.reset_all()

    # ------------------------------------------------------------------------------------------------ front-end
    def accept_wave(self, pcm):
        """:335-398 with int16 samples (a numpy array / list) instead of bytes; None = not enough samples yet."""
        wave = np.append(self.wave_remained, np.asarray(pcm, dtype=np.int64))            # :346-347
        if wave.size < (self.frame_length * self.sample_rate / 1000) * self.right_context:
            self.wave_remained = wave                                                     # :348-351
            return None
        wave_tensor = torch.from_numpy(wave).float()
        if self.fbank_fn is not None:
            feats = self.fbank_fn(wave_tensor)
        else:                                                                             # :352-360
            feats = O.fbank(wave_tensor, num_mel_bins=self.num_mel_bins, frame_length=self.frame_length,
                            frame_shift=self.frame_shift)
        feat_len = len(feats)
        frame_shift = int(self.frame_shift / 1000 * self.sample_rate)
        self.wave_remained = wave[feat_len * frame_shift:]                                # :362-364
        if self.context_expansion:                                                        # :366-390
            if not feat_len > self.right_context:
                raise ValueError("make sure each chunk feat length is large than right context.")
            if self.feature_remained is None:
                feats_pad = F.pad(feats.T, (self.left_context, 0), mode='replicate').T
            else:
                feats_pad = torch.cat((self.feature_remained, feats))
            ctx_frm = feats_pad.shape[0] - (self.right_context + self.right_context)
            ctx_win = self.left_context + self.right_context + 1
            feats_ctx = torch.zeros(ctx_frm, feats.shape[1] * ctx_win, dtype=torch.float32)
            for i in range(ctx_frm):
                feats_ctx[i] = torch.cat(tuple(feats_pad[i:i + ctx_win])).unsqueeze(0)
            self.feature_remained = feats[-(self.left_context + self.right_context):]
            feats = feats_ctx
        if self.downsampling > 1:                                                         # :391-397
            last_remainder = 0 if self.feats_ctx_offset == 0 else self.downsampling - self.feats_ctx_offset
            remainder = (feats.size(0) + last_remainder) % self.downsampling
            feats = feats[self.feats_ctx_offset::self.downsampling, :]
            self.feats_ctx_offset = remainder if remainder == 0 else self.downsampling - remainder
        return feats

    # ------------------------------------------------------------------------------------------------ decoding
    def execute_detection(self, t):
        """:411-480 (the log-only branches left out)."""
        hit_keyword, start, end = None, 0, 0
        hyps = [(y[0], y[1][0] + y[1][1], y[1][2]) for y in self.cur_hyps]
        for one_hyp in hyps:
            prefix_ids, prefix_nodes = one_hyp[0], one_hyp[2]
            for word in self.keywords_token.keys():
                lab = self.keywords_token[word]['token_id']
                offset = O.is_sublist(prefix_ids, lab)
                if offset != -1:
                    hit_keyword = word
                    start = prefix_nodes[offset]['frame']
                    end = prefix_nodes[offset + len(lab) - 1]['frame']
                    for idx in range(offset, offset + len(lab)):
                        self.hit_score *= prefix_nodes[idx]['prob']
                    break
            if hit_keyword is not None:
                self.hit_score = math.sqrt(self.hit_score)
                break
        duration = end - start
        if hit_keyword is not None:
            if self.hit_score >= self.threshold and self.min_frames <= duration <= self.max_frames \
                    and (self.last_active_pos == -1 or end - self.last_active_pos >= self.interval_frames):
                self.activated = True
                self.last_active_pos = end
        self.result = {
            "state": 1 if self.activated else 0,
            "keyword": hit_keyword if self.activated else None,
            "start": start * self.resolution if self.activated else None,
            "end": end * self.resolution if self.activated else None,
            "score": self.hit_score if self.activated else None,
        }

    def forward_probs(self, probs):
        """:489-514 for one chunk of softmax posteriors (T, V)."""
        if probs.size(0) < 1:
            return {}
        for t, prob in enumerate(probs):
            t *= self.downsampling
            # decode_keywords :400-409: one frame of the streaming search, then keep path_beam hypotheses
            self.cur_hyps = O.ctc_prefix_beam_search(prob.unsqueeze(0), self.keywords_idxset, self.score_beam,
                                                     self.path_beam, cur_hyps=self.cur_hyps,
                                                     frame_offset=t + self.total_frames)
            self.execute_detection(t)
            if self.activated:
                self.reset()
                break
        self.total_frames += len(probs) * self.downsampling
        if len(self.cur_hyps) > 0 and len(self.cur_hyps[0][0]) > 0:
            keyword_may_start = int(self.cur_hyps[0][1][2][0]['frame'])
            if (self.total_frames - keyword_may_start) > self.max_frames:
                self.reset()
        return self.result

    def forward(self, pcm):
        """:482-514: one chunk of int16 samples -> the result dict ({} = no feature rows)."""
        feature = self.accept_wave(pcm)
        if feature is None or feature.size(0) < 1:
            return {}
        logits, self.in_cache = self.model_fn(feature.unsqueeze(0), self.in_cache)
        return self.forward_probs(logits.softmax(2)[0])

    def reset(self):
        self.cur_hyps = [(tuple(), (1.0, 0.0, []))]
        self.activated = False
        self.hit_score = 1.0

    def reset_all(self):
        self.reset()
        self.wave_remained = np.array([])
        self.feature_remained = None
        self.feats_ctx_offset = 0
        self.in_cache = torch.zeros(0, 0, 0, dtype=torch.float)
        self.total_frames = 0
        self.last_active_pos = -1
        self.result = {}
