"""Batched streaming CTC keyword spotter: int16 PCM chunks in, detections out, decoded on the GPU.

The reference's ``KeyWordSpotter`` (``wekws/bin/stream_kws_ctc.py:218-529``) runs one stream: it carries PCM and feature
rows from chunk to chunk (``accept_wave`` :335-398), runs the model with its cache, and after every frame one step of
the prefix beam search plus ``execute_detection`` (:411-480).  This class does the same for ``num_streams`` streams per
call, bit-exact in its results (``state``, ``keyword``, ``start``, ``end`` equal, ``score`` the same double):

* splice + Fbank, context expansion + frame skip and decode + detect are kernels of csrc/kws_stream.cu (the Fbank and
  the model are the library's own); per-stream row counts and offsets are planned here from sample counts, so no call
  reads anything back to plan the next;
* streams may get different row counts in one call (ragged ``lengths``, a ``reset_all`` of some streams): they are
  grouped by row count and the model runs once per group, its cache gathered / scattered along the batch dimension;
* ``forward`` copies the results to the host once per call; ``forward_async`` returns them on the device.

Token ids are given directly (``{word: {"token_id": [...]}}``); the reference's token / lexicon file parsers are not
part of this package.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import _native
from .ctc import MAX_PATH_BEAM, MAX_SCORE_BEAM
from .frontend import Fbank

SAMPLE_RATE = 16000


class StreamPlanner:
    """The host half of accept_wave (:335-398) for B streams: per-stream sample / row counts as integers.  No CUDA --
    every kernel argument of a call follows from the sample counts, so nothing is read back from the device."""

    def __init__(self, num_streams: int, frame_length=25, frame_shift=10, context=None, frame_skip: int = 1):
        self.B = int(num_streams)
        self.win = int(frame_length * SAMPLE_RATE / 1000)
        self.shift = int(frame_shift / 1000 * SAMPLE_RATE)                         # :363
        self.expand = context is not None
        self.left, self.right = (int(context[0]), int(context[1])) if self.expand else (0, 0)
        if self.expand and (self.left < 0 or self.right < 0 or self.left + self.right < 1 or self.left > self.right):
            raise ValueError("context must be (left, right) with 0 <= left <= right and left + right >= 1")
        self.skip = int(frame_skip)
        if self.skip < 1:
            raise ValueError("frame_skip must be >= 1")
        self.min_wave = frame_length * SAMPLE_RATE / 1000 * self.right   # :348-349: below this the wave is carried
        self.carry_cap = max(self.win - 1, self.win * self.right - 1)    # the longest PCM carry that can occur
        self.carry_len = np.zeros(self.B, dtype=np.int64)                # samples carried (wave_remained)
        self.fc_len = -np.ones(self.B, dtype=np.int64)                   # feature rows carried, -1 = None (first chunk)
        self.skip_off = np.zeros(self.B, dtype=np.int64)                 # feats_ctx_offset

    def reset_all(self, ids) -> None:
        self.carry_len[ids] = 0
        self.fc_len[ids] = -1
        self.skip_off[ids] = 0

    def plan(self, new_len) -> dict:
        """One call with new_len[b] new samples per stream.  Raises ValueError (nothing changed) if a stream would hit
        the reference's `feat_len > right_context` assert (:367-368).  `rows` = model rows per stream (0: the reference
        returns {}); commit() makes the carries the plan computed current."""
        new_len = np.asarray(new_len, dtype=np.int64)
        wave = self.carry_len + new_len                               # :347
        run = wave >= self.min_wave                                   # :348-351
        nf = np.where(run & (wave >= self.win), 1 + (wave - self.win) // self.shift, 0)
        consumed = nf * self.shift                                    # :364
        fc_after = self.fc_len.copy()
        if self.expand:
            bad = run & (nf <= self.right)
            if bad.any():
                raise ValueError(f"streams {np.nonzero(bad)[0].tolist()}: a chunk gives {nf[bad].tolist()} feature rows, "
                                 f"not more than the right context {self.right} (stream_kws_ctc.py:367)")
            x = np.where(self.fc_len < 0, self.left, self.fc_len) + nf - 2 * self.right   # :378-379, right + right
            if (run & (x < 0)).any():
                raise ValueError("a chunk gives a negative number of context rows (stream_kws_ctc.py:378-382)")
            fc_after = np.where(run, np.minimum(nf, self.left + self.right), self.fc_len)  # :388-389
        else:
            x = nf
        x = np.where(run, x, 0)
        off_after = self.skip_off.copy()
        if self.skip > 1:                                             # :391-397
            o = self.skip_off
            rows = np.where(x > o, (x - o + self.skip - 1) // self.skip, 0)
            last_rem = np.where(o == 0, 0, self.skip - o)
            rem = (x + last_rem) % self.skip
            off_after = np.where(run, np.where(rem == 0, 0, self.skip - rem), o)
        else:
            rows = x
        rows = np.where(run, rows, 0)
        return dict(new_len=new_len, wave=wave, run=run, nf=nf, consumed=consumed, carry_after=wave - consumed,
                    fc_after=fc_after, off_after=off_after, rows=rows)

    def commit(self, p: dict) -> None:
        self.carry_len, self.fc_len, self.skip_off = p["carry_after"], p["fc_after"], p["off_after"]


class KeyWordSpotter:
    """``KeyWordSpotter(model, keywords_token, threshold, num_streams, device, ...)``; see the module docstring.

    model: a CTC ``KWSModel`` (``init_model``) whose input dim is num_mel_bins * (left + right + 1).  context: None (no
    context expansion) or (left, right) with left <= right (the reference's row count formula fails for left > right).
    """

    def __init__(self, model, keywords_token: Dict[str, dict], threshold: float, num_streams: int, device,
                 num_mel_bins: int = 80, frame_length: int = 25, frame_shift: int = 10, context=None,
                 frame_skip: int = 1, min_frames: int = 5, max_frames: int = 250, interval_frames: int = 50,
                 score_beam: int = 3, path_beam: int = 20):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("wekws_b200.KeyWordSpotter runs on CUDA (sm_100a) only (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if not 1 <= score_beam <= MAX_SCORE_BEAM or not 1 <= path_beam <= MAX_PATH_BEAM:
            raise ValueError(f"score_beam must be in 1..{MAX_SCORE_BEAM} and path_beam in 1..{MAX_PATH_BEAM}")
        self.model = model
        self.B = int(num_streams)
        self.num_mel_bins = int(num_mel_bins)
        self.frame_length, self.frame_shift = frame_length, frame_shift
        self.resolution = frame_shift / 1000                                      # :251
        self.planner = pl = StreamPlanner(num_streams, frame_length, frame_shift, context, frame_skip)
        self.expand, self.left, self.right, self.skip = pl.expand, pl.left, pl.right, pl.skip
        self.idim = self.num_mel_bins * (self.left + self.right + 1)
        if model.idim != self.idim:
            raise ValueError(f"model input_dim {model.idim} != num_mel_bins x context window = {self.idim}")
        self.cfg = _native.KwsConfig(float(threshold), int(min_frames), int(max_frames), int(interval_frames),
                                     int(score_beam), int(path_beam), self.skip)
        self.threshold = threshold
        self.fbank = Fbank(self.num_mel_bins, float(frame_length), float(frame_shift), device=self.device)
        self._cache_dim = 1 if isinstance(model.backbone, nn.GRU) else 0
        lib = _native.lib()
        dev, B = self.device, self.B
        self.state = torch.zeros(B, int(lib.wekws_kws_state_bytes()), dtype=torch.uint8, device=dev)
        self._pcm_carry = torch.zeros(2, B, max(pl.carry_cap, 1), dtype=torch.int16, device=dev)
        C_rows = self.left + self.right
        self._feat_carry = torch.zeros(2, B, max(C_rows, 1), self.num_mel_bins, dtype=torch.float32, device=dev)
        self._parity = 0
        with torch.cuda.device(dev):
            _, self.cache = model(torch.zeros(B, 0, self.idim, device=dev))       # zeros == the reference's _EMPTY
        self.overflow = np.zeros(B, dtype=bool)
        self.features = self.probs = self.row_offsets = self.rows = None
        self.stage_hook = None        # callable(stage name) at each stage boundary of forward_async (timing)
        self.set_keywords(keywords_token)
        self.reset_all()

    @classmethod
    def from_configs(cls, configs: dict, model, keywords_token, threshold, num_streams, device, **gates):
        """Front-end settings from a training config's ``dataset_conf`` in either schema: the legacy
        ``feature_extraction_conf`` the reference script reads (:239-259), or ``fbank_conf`` + ``context_expansion`` /
        ``context_expansion_conf`` + ``frame_skip`` as the shipped CTC configs have it."""
        dc = configs["dataset_conf"]
        fe = dc.get("feature_extraction_conf") or dc.get("fbank_conf")
        if fe is None:
            raise ValueError("dataset_conf has neither feature_extraction_conf nor fbank_conf")
        context = None
        if dc.get("context_expansion", False):
            cc = dc["context_expansion_conf"]
            context = (cc["left"], cc["right"])
        return cls(model, keywords_token, threshold, num_streams, device, num_mel_bins=fe["num_mel_bins"],
                   frame_length=fe["frame_length"], frame_shift=fe["frame_shift"], context=context,
                   frame_skip=dc.get("frame_skip", 1), **gates)

    def set_keywords(self, keywords_token: Dict[str, dict]) -> None:
        """set_keywords :304-333 with token ids given: keywords in dict order, token set = {0} | every keyword's ids."""
        if not keywords_token:
            raise ValueError("at least one keyword is needed")
        self.words = list(keywords_token.keys())
        seqs = [[int(t) for t in keywords_token[w]["token_id"]] for w in self.words]
        if any(len(s) == 0 for s in seqs):
            raise ValueError("every keyword needs at least one token")
        idxset = {0}
        for s in seqs:
            idxset.update(s)
        offs = [0]
        for s in seqs:
            offs.append(offs[-1] + len(s))
        dev = self.device
        self._tokset = torch.tensor(sorted(idxset), dtype=torch.int32, device=dev)
        self._kw_tokens = torch.tensor([t for s in seqs for t in s], dtype=torch.int32, device=dev)
        self._kw_offs = torch.tensor(offs, dtype=torch.int32, device=dev)

    # ---------------------------------------------------------------------------------------------------- resets
    def _ids(self, streams):
        if streams is None:
            return list(range(self.B))
        ids = [int(s) for s in streams]
        if any(not 0 <= s < self.B for s in ids):
            raise IndexError("stream index out of range")
        return ids

    def _reset_device(self, ids: List[int], full: bool) -> None:
        if not ids:
            return
        d_ids = None
        if len(ids) != self.B or ids != list(range(self.B)):
            d_ids = torch.tensor(ids, dtype=torch.int32).pin_memory().to(self.device, non_blocking=True)
        with torch.cuda.device(self.device):
            rc = _native.lib().wekws_kws_reset(
                C.c_void_p(self.state.data_ptr()), self.B, None if d_ids is None else C.c_void_p(d_ids.data_ptr()),
                len(ids), 1 if full else 0, C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream))
        _native.check(rc, "wekws_kws_reset")
        if full:
            if d_ids is None:
                self.cache.zero_()
            else:
                self.cache.index_fill_(self._cache_dim, d_ids.long(), 0.0)

    def reset(self, streams: Optional[Sequence[int]] = None) -> None:
        """reset() :516-519: initial beam, activated = False, hit_score = 1.0."""
        self._reset_device(self._ids(streams), False)

    def reset_all(self, streams: Optional[Sequence[int]] = None) -> None:
        """reset_all() :521-529: also the PCM / feature carries, the frame-skip offset, the model cache, total_frames
        and last_active_pos."""
        ids = self._ids(streams)
        self.planner.reset_all(ids)
        self._reset_device(ids, True)

    # ---------------------------------------------------------------------------------------------------- forward
    def forward_async(self, pcm: torch.Tensor, lengths: Optional[Sequence[int]] = None) -> torch.Tensor:
        """One chunk per stream: pcm (B, N) int16 CUDA, lengths (host ints, default N) the valid samples per row.
        Returns the (B, 6) int64 device results (see include/wekws_b200.h wekws_kws_detect); no host synchronisation."""
        if not pcm.is_cuda or pcm.dtype != torch.int16 or pcm.dim() != 2 or pcm.size(0) != self.B:
            raise ValueError(f"pcm must be a ({self.B}, N) int16 CUDA tensor")
        if pcm.device != self.device:
            raise ValueError(f"pcm is on {pcm.device}, the spotter on {self.device}")
        if pcm.stride(1) != 1:
            pcm = pcm.contiguous()
        N = pcm.size(1)
        new_len = np.full(self.B, N, dtype=np.int64) if lengths is None else np.asarray(lengths, dtype=np.int64)
        if new_len.shape != (self.B,) or (new_len < 0).any() or (new_len > N).any():
            raise ValueError("lengths must be B host integers in 0..N")
        pl = self.planner
        p = pl.plan(new_len)
        B, dev, lib = self.B, self.device, _native.lib()
        rows = p["rows"]
        # streams grouped by row count (0 rows: not part of any model call), rows packed group after group
        order = sorted((int(b) for b in np.nonzero(rows)[0]), key=lambda b: (int(rows[b]), b))
        row_off = np.zeros(B, dtype=np.int64)
        groups, cur = [], 0
        for b in order:
            if not groups or groups[-1][0] != rows[b]:
                groups.append([int(rows[b]), cur, []])
            groups[-1][2].append(b)
            row_off[b] = cur
            cur += int(rows[b])
        R = cur
        # one host -> device copy of the whole plan
        cols = [new_len, pl.carry_len, p["consumed"], np.where(p["run"], p["wave"], 0), p["nf"], pl.fc_len,
                pl.skip_off, row_off, rows, np.asarray(order + [0] * (B - len(order)), dtype=np.int64)]
        host = torch.from_numpy(np.stack(cols).astype(np.int32)).pin_memory()
        d = host.to(dev, non_blocking=True)
        d_new, d_carry, d_cons, d_flen, d_nf, d_fcl, d_off, d_roff, d_rows, d_perm = d.unbind(0)

        def ptr(t):
            return C.c_void_p(t.data_ptr())

        with torch.cuda.device(dev):
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            src, dst = self._parity, 1 - self._parity
            mark = self.stage_hook or (lambda name: None)
            mark("splice_fbank")
            S = (int(p["wave"].max()) + 7) // 8 * 8 if B else 0     # 16-byte rows: the Fbank's vector loads
            stage = torch.empty(B, max(S, 1), dtype=torch.int16, device=dev)
            _native.check(lib.wekws_kws_splice(
                ptr(pcm), pcm.stride(0), ptr(d_new), ptr(d_carry), ptr(d_cons), ptr(self._pcm_carry[src]),
                ptr(self._pcm_carry[dst]), self._pcm_carry.size(2), ptr(stage), S, B, stream), "wekws_kws_splice")
            feats = self.fbank(stage[:, :S], lengths=d_flen)
            T = feats.size(1)
            mark("context")
            x = torch.empty(max(R, 1), self.idim, dtype=torch.float32, device=dev)
            _native.check(lib.wekws_kws_context(
                ptr(feats) if feats.numel() else None, B, T, self.num_mel_bins, ptr(d_nf),
                ptr(self._feat_carry[src]), ptr(d_fcl), ptr(self._feat_carry[dst]), self.left, self.right,
                1 if self.expand else 0, self.skip, ptr(d_off), ptr(d_roff), ptr(d_rows), int(rows.max()) if B else 0,
                ptr(x), stream), "wekws_kws_context")
            mark("model")
            probs = self._model_groups(x, groups, d_perm, B) if R else x
            mark("decode_detect")
            result = torch.empty(B, _native.KWS_RESULT_FIELDS, dtype=torch.int64, device=dev)
            _native.check(lib.wekws_kws_detect(
                ptr(probs), ptr(d_roff), ptr(d_rows), B, self.model.odim, ptr(self._tokset), self._tokset.numel(),
                ptr(self._kw_tokens), ptr(self._kw_offs), len(self.words), C.byref(self.cfg), ptr(self.state),
                ptr(result), stream), "wekws_kws_detect")
            mark("end")
        self._parity = dst
        pl.commit(p)
        # the last call's model input / posteriors, stream b at packed rows row_offsets[b] .. + rows[b] (inspection)
        self.features, self.probs, self.row_offsets, self.rows = x[:R], probs[:R], row_off, rows
        return result

    def _model_groups(self, x, groups, d_perm, B):
        """model.forward_softmax once per row-count group; the cache is gathered / scattered along its batch dim."""
        outs, first = [], 0
        for T, start, members in groups:
            nb = len(members)
            xg = x[start:start + nb * T].view(nb, T, self.idim)
            if nb == B:          # every stream, in stream order (a single group is sorted by stream index)
                y, self.cache = self.model.forward_softmax(xg, self.cache)
            else:
                idx = d_perm[first:first + nb].long()
                y, c = self.model.forward_softmax(xg, self.cache.index_select(self._cache_dim, idx))
                self.cache.index_copy_(self._cache_dim, idx, c)
            outs.append(y.view(nb * T, -1))
            first += nb
        return outs[0] if len(outs) == 1 else torch.cat(outs)

    def results(self, result: torch.Tensor) -> List[dict]:
        """Device results of forward_async -> the reference's dicts (one device-to-host copy)."""
        r = result.cpu().numpy()
        score = r[:, 4].copy().view(np.float64)
        out = []
        for b in range(r.shape[0]):
            st = int(r[b, 0])
            if st < 0:
                out.append({})
            elif st == 0:
                out.append({"state": 0, "keyword": None, "start": None, "end": None, "score": None})
            else:
                out.append({"state": 1, "keyword": self.words[int(r[b, 1])], "start": int(r[b, 2]) * self.resolution,
                            "end": int(r[b, 3]) * self.resolution, "score": float(score[b])})
        self.overflow = r[:, 5].astype(bool)
        return out

    def forward(self, pcm: torch.Tensor, lengths: Optional[Sequence[int]] = None) -> List[dict]:
        """forward() :482-514 for every stream: the reference's result dict per stream ({} = no feature rows yet).
        After the call ``self.overflow[b]`` is True if stream b's hypotheses outgrew the device limits (results of that
        stream are then not exact; reset_all clears it)."""
        return self.results(self.forward_async(pcm, lengths))

    __call__ = forward
