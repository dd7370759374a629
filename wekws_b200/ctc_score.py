"""Test-set scoring and DET statistics of the CTC recipes on the GPU (run_ctc.sh / run_fsmn_ctc.sh stage 3).

* ``ctc_stream_score`` + ``write_ctc_stream_scores`` replace the per-utterance, per-frame pure-Python decode of
  ``wekws/bin/stream_score_ctc.py:209-381`` with one kernel launch over a batch (csrc/ctc_score.cu), and write the
  same score file bytes.
* ``compute_det_ctc`` replaces ``wekws/bin/compute_det_ctc.py``: the label / score join (:50-124) on the host, the
  threshold sweep (:251-281) with one kernel launch per keyword, the same ``stats.<keyword>.txt`` bytes.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, Iterable, List, Optional, Sequence

import torch

from . import _native
from .ctc import MAX_PREFIX
from .postproc import det_thresholds


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _keyword_tensors(keywords_token: Dict[str, dict], dev):
    """Keyword token sequences back to back + offsets (dict order) and keywords_idxset = {0} | their tokens
    (stream_score_ctc.py:188-199)."""
    seqs = [[int(t) for t in keywords_token[w]["token_id"]] for w in keywords_token]
    if not seqs or any(len(s) == 0 for s in seqs):
        raise ValueError("keywords_token needs at least one keyword, each with at least one token")
    offs = [0]
    for s in seqs:
        offs.append(offs[-1] + len(s))
    flat = torch.tensor([t for s in seqs for t in s], dtype=torch.int32, device=dev)
    idxset = torch.tensor(sorted({0} | {t for s in seqs for t in s}), dtype=torch.int32, device=dev)
    return flat, torch.tensor(offs, dtype=torch.int32, device=dev), idxset


class CtcStreamScores:
    """Device result of ctc_stream_score: count (B,) int32 activations, overflow (B,) int32, and the first
    max_detections activations of each utterance in frame order: keyword (B, D) int32 (index into ``words``),
    score (B, D) float64 hit_score, start / end (B, D) int32 frames."""

    def __init__(self, B, max_detections, words, dev):
        self.B, self.max_detections, self.words = B, max_detections, list(words)
        self.count = torch.empty(B, dtype=torch.int32, device=dev)
        self.overflow = torch.empty(B, dtype=torch.int32, device=dev)
        self.keyword = torch.empty(B, max_detections, dtype=torch.int32, device=dev)
        self.score = torch.empty(B, max_detections, dtype=torch.float64, device=dev)
        self.start = torch.empty(B, max_detections, dtype=torch.int32, device=dev)
        self.end = torch.empty(B, max_detections, dtype=torch.int32, device=dev)


def ctc_stream_score(probs: torch.Tensor, lengths, keywords_token: Dict[str, dict], threshold: float = 0.0,
                     min_frames: int = 5, max_frames: int = 250, score_beam_size: int = 3, path_beam_size: int = 20,
                     frame_skip: int = 1, max_detections: int = 16) -> CtcStreamScores:
    """stream_score_ctc.py:221-377 for a batch, one kernel launch.  probs (B, T, V) float32 CUDA softmax of
    ``model(feats)`` (:218-219); lengths (B,) valid rows (``feats_lengths`` after the model; None = T);
    keywords_token {word: {'token_id': [...]}} in the script's dict order; frame_skip = dataset_conf.frame_skip.
    The defaults are the script's argparse defaults."""
    if not probs.is_cuda:
        raise RuntimeError("wekws_b200.ctc_stream_score runs on CUDA only; got a CPU tensor (no CPU fallback)")
    if probs.dim() != 3 or probs.dtype != torch.float32:
        raise ValueError("probs must be a (B, T, V) float32 tensor")
    if max_detections < 1:
        raise ValueError("max_detections must be >= 1")
    probs = probs.contiguous()
    B, T, V = probs.shape
    dev = probs.device
    lens = None
    if lengths is not None:
        lens = torch.as_tensor(lengths).to(device=dev, dtype=torch.int32).contiguous()
        if tuple(lens.shape) != (B,):
            raise ValueError(f"lengths must have shape ({B},)")
        if B and (int(lens.min()) < 0 or int(lens.max()) > T):
            raise ValueError(f"lengths must lie in [0, {T}]")
    words = list(keywords_token)
    flat, offs, idxset = _keyword_tensors(keywords_token, dev)
    out = CtcStreamScores(B, int(max_detections), words, dev)
    cfg = _native.CtcScoreConfig(float(threshold), int(min_frames), int(max_frames), int(score_beam_size),
                                 int(path_beam_size), int(frame_skip), int(max_detections))
    with torch.cuda.device(dev):
        rc = _native.lib().wekws_ctc_stream_score(
            _ptr(probs), _ptr(lens), B, T, V, _ptr(idxset), idxset.numel(), _ptr(flat), _ptr(offs), len(words),
            C.byref(cfg), _ptr(out.count), _ptr(out.overflow), _ptr(out.keyword), _ptr(out.score), _ptr(out.start),
            _ptr(out.end), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _native.check(rc, "wekws_ctc_stream_score")
    return out


def write_ctc_stream_scores(fout, keys: Sequence[str], scores: CtcStreamScores, words: Optional[Sequence[str]] = None):
    """The score lines of stream_score_ctc.py:349-350,375-376: '{key} detected {keyword} {score:.3f}' per activation
    in frame order, or '{key} rejected'.  One device-to-host copy.  Raises (naming the keys) if an utterance
    overflowed the decoder or had more than max_detections activations: the file would not be the script's."""
    words = scores.words if words is None else list(words)
    if len(keys) != scores.B:
        raise ValueError(f"{len(keys)} keys for {scores.B} utterances")
    D = scores.max_detections
    ints = torch.cat([scores.count.view(-1, 1), scores.overflow.view(-1, 1), scores.keyword], 1).to(torch.float64)
    host = torch.cat([ints, scores.score], 1).cpu()             # int32 values are exact in float64
    count = host[:, 0].long().tolist()
    overflow = host[:, 1].long().tolist()
    kw = host[:, 2:2 + D].long().tolist()
    sc = host[:, 2 + D:].tolist()
    bad = [keys[b] for b in range(scores.B) if overflow[b] or count[b] > D]
    if bad:
        raise RuntimeError(f"wekws_b200.write_ctc_stream_scores: {len(bad)} utterance(s) overflowed the decoder "
                           f"(prefix > {MAX_PREFIX} tokens or node pool full) or had more than max_detections={D} "
                           f"activations: {', '.join(bad[:20])}{' ...' if len(bad) > 20 else ''}")
    for b, key in enumerate(keys):
        if count[b] == 0:
            fout.write('{} rejected\n'.format(key))
        for i in range(count[b]):
            fout.write('{} detected {} {:.3f}\n'.format(key, words[kw[b][i]], sc[b][i]))


# ------------------------------------------------------------------------------------------------ compute_det_ctc
_LATIN_RUN = re.compile(r"[A-Za-z!?,<>()']+")


def split_mixed_label(text: str) -> List[str]:
    """compute_det_ctc.py:30-41: lower-cased; a run of Latin letters (and !?,<>()') is one token, any other character
    is one token; spaces between tokens are dropped."""
    tokens = []
    rest = text.lower()
    while rest:
        m = _LATIN_RUN.match(rest)
        tok = m.group(0) if m is not None else rest[0]
        tokens.append(tok)
        rest = rest[len(tok):].strip(' ')
    return tokens


def space_mixed_label(text: str) -> str:
    """compute_det_ctc.py:44-47: the tokens of split_mixed_label joined by single spaces."""
    return ' '.join(split_mixed_label(text)).strip()


def ctc_det_tables(label_list: Iterable[dict], score_lines: Iterable[str], true_keywords: Dict[str, str]):
    """load_label_and_score of compute_det_ctc.py:50-124.  label_list: data.list objects (key, txt, duration) in file
    order; score_lines: the score file's lines; true_keywords {keyword: token string}.  Returns
    {spaced keyword: {'keyword_table': {key: confi}, 'keyword_duration', 'filler_table', 'filler_duration'}} in
    keyword order, durations summed in label order."""
    scores = {}
    for line in score_lines:
        arr = line.strip().split()
        key = arr[0]
        if arr[1] == 'detected':
            kw = true_keywords[arr[2]]
            if key not in scores:                       # the first line of a key wins
                scores[key] = (space_mixed_label(kw), float(arr[3]))
        elif key not in scores:
            scores[key] = ('unknown', -1.0)
    spaced = [space_mixed_label(true_keywords[k]) for k in true_keywords]
    tables = {}
    for kw in spaced:
        tables[kw] = {'keyword_table': {}, 'keyword_duration': 0.0, 'filler_table': {}, 'filler_duration': 0.0}
    for obj in label_list:
        for field in ('key', 'txt', 'duration'):
            if field not in obj:
                raise ValueError(f"label object without '{field}': {obj}")
        key = obj['key']
        if key not in scores:
            raise KeyError(f"label key {key!r} has no line in the score file")
        txt = ' ' + space_mixed_label(obj['txt']) + ' '
        got_kw, confi = scores[key]
        for kw in spaced:
            side = 'keyword' if txt.find(' ' + kw + ' ') != -1 else 'filler'
            tables[kw][side + '_table'][key] = confi if kw == got_kw else -1.0
            tables[kw][side + '_duration'] += obj['duration']
    return tables


def ctc_det_sweep(conf_kw: torch.Tensor, conf_filler: torch.Tensor, thresholds: torch.Tensor):
    """compute_det_ctc.py:251-270 for one keyword on the device: (false_reject, false_alarm) int64 CUDA tensors of
    #(conf_kw < thr) and #(conf_filler >= thr) per threshold.  Inputs are float64 CUDA tensors."""
    for t in (conf_kw, conf_filler, thresholds):
        if not t.is_cuda or t.dtype != torch.float64 or t.dim() != 1:
            raise ValueError("ctc_det_sweep takes 1-D float64 CUDA tensors (no CPU fallback)")
    conf_kw, conf_filler, thresholds = conf_kw.contiguous(), conf_filler.contiguous(), thresholds.contiguous()
    dev = thresholds.device
    fr = torch.empty(thresholds.numel(), dtype=torch.int64, device=dev)
    fa = torch.empty_like(fr)
    with torch.cuda.device(dev):
        rc = _native.lib().wekws_ctc_det_sweep(
            _ptr(conf_kw), conf_kw.numel(), _ptr(conf_filler), conf_filler.numel(), _ptr(thresholds),
            thresholds.numel(), _ptr(fr), _ptr(fa), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    _native.check(rc, "wekws_ctc_det_sweep")
    return fr, fa


def compute_det_ctc(label_list: Iterable[dict], score_lines: Iterable[str], true_keywords: Dict[str, str],
                    step: float = 0.01, stats_dir: Optional[str] = None, device="cuda"):
    """compute_det_ctc.py without the plot: returns {spaced keyword: [(threshold, false_alarm_per_hour,
    false_reject_rate), ...]} and, with stats_dir, writes stats.<keyword with spaces as _>.txt rows
    '{:.3f} {:.6f} {:.6f}' there, the script's bytes."""
    tables = ctc_det_tables(label_list, score_lines, true_keywords)
    thr = det_thresholds(step)
    d_thr = thr.to(device)
    out = {}
    for kw, tab in tables.items():
        keyword_num, filler_num = len(tab['keyword_table']), len(tab['filler_table'])
        if keyword_num == 0:
            raise ValueError(f"Can't compute det for {kw} without positive sample")
        if filler_num == 0:
            raise ValueError(f"Can't compute det for {kw} without negative sample")
        ck = torch.tensor(list(tab['keyword_table'].values()), dtype=torch.float64).to(device)
        cf = torch.tensor(list(tab['filler_table'].values()), dtype=torch.float64).to(device)
        fr, fa = ctc_det_sweep(ck, cf, d_thr)
        counts = torch.stack([fr, fa]).cpu().tolist()
        filler_dur = tab['filler_duration']
        rows = []
        for i, th in enumerate(thr.tolist()):
            rows.append((th, max(counts[1][i], 1e-6) / (filler_dur / 3600.0), counts[0][i] / keyword_num))
        out[kw] = rows
        if stats_dir is not None:
            with open(os.path.join(stats_dir, 'stats.' + kw.replace(' ', '_') + '.txt'), 'w', encoding='utf8') as f:
                for row in rows:
                    f.write('{:.3f} {:.6f} {:.6f}\n'.format(*row))
    return out
