"""CPU oracle of the CTC recipes' evaluation scripts (stage 3 of run_ctc.sh / run_fsmn_ctc.sh).

TEST INFRASTRUCTURE ONLY.  It restates, statement for statement, what the reference does (line numbers of
wekws/bin/stream_score_ctc.py and wekws/bin/compute_det_ctc.py):

* stream_score        stream_score_ctc.py:221-377   one utterance's per-frame decode and detection -> score lines
* split_mixed_label   compute_det_ctc.py:30-47      (and space_mixed_label)
* load_label_and_score compute_det_ctc.py:50-124    the label / score join
* det_stats_text      compute_det_ctc.py:228-281    one stats.<keyword>.txt per keyword (no plot)
* plant_logits        CTC-like test logits (the golden generator, the GPU tests and scripts/bench_ctc_score.py)

The beam step is kws_oracle.ctc_prefix_beam_search (pinned by tests/golden/ctc.npz); this module is pinned by
tests/golden/ctc_score.npz, which oracle/make_ctc_score_golden.py makes by running the reference scripts.
"""
from __future__ import annotations

import math
import re

import torch

from . import kws_oracle as O


def _frame_is_skipped(prob, idxset, score_beam):
    """:243-261: top-k, then `prob > 0.05 and idx in keywords_idxset`; True when nothing is left."""
    top_p, top_i = prob.topk(score_beam)
    return not any(p > 0.05 and i in idxset for p, i in zip(top_p.tolist(), top_i.tolist()))


def stream_score(key, probs, keywords_token, threshold=0.0, min_frames=5, max_frames=250, score_beam=3, path_beam=20,
                 frame_skip=1, events=None):
    """Score lines of one utterance.  probs (n, V) float32 softmax rows (logits[i][:lengths[i]], :223);
    keywords_token {word: {'token_id': (...)}} in dict order.  Returns (lines, detections) with detections
    [(word, hit_score, start, end)] in frame order.  events (a dict) counts what happened, for coverage checks:
    skipped frames, threshold rejections, carried_sqrt (a frame with a carried hit and no keyword in hyps[0]) and
    stale_duration (a duration rejection on such a frame)."""
    events = {} if events is None else events

    def count(what):
        events[what] = events.get(what, 0) + 1
    idxset = {0}
    for w in keywords_token:
        idxset.update(keywords_token[w]['token_id'])
    cur_hyps = [(tuple(), (1.0, 0.0, []))]                                  # :228
    hit_keyword, hit_score, start, end = None, 1.0, 0, 0                    # :230-234
    detections = []
    for row in range(probs.size(0)):                                        # :237
        t = row * frame_skip                                                # :239
        if _frame_is_skipped(probs[row], idxset, score_beam):
            count('skipped')
            continue                                                        # :260-261
        cur_hyps = O.ctc_prefix_beam_search(probs[row:row + 1], idxset, score_beam, path_beam, cur_hyps=cur_hyps,
                                            frame_offset=t)                 # :263-319
        carried, found = hit_keyword is not None, False
        for prefix_ids, _, prefix_nodes in O.hyps_of(cur_hyps):            # :321-342
            for word in keywords_token:
                lab = keywords_token[word]['token_id']
                offset = O.is_sublist(prefix_ids, lab)
                if offset != -1:
                    found = True
                    hit_keyword = word
                    start = prefix_nodes[offset]['frame']
                    end = prefix_nodes[offset + len(lab) - 1]['frame']
                    for idx in range(offset, offset + len(lab)):
                        hit_score *= prefix_nodes[idx]['prob']
                    break
            if hit_keyword is not None:                                     # also a hit carried from an earlier frame
                hit_score = math.sqrt(hit_score)
                break
        duration = end - start                                              # :344-360
        if carried and not found and cur_hyps:
            count('carried_sqrt')
        if hit_keyword is not None and hit_score < threshold:
            count('threshold_reject')
        elif hit_keyword is not None and not min_frames <= duration <= max_frames and not found:
            count('stale_duration')
        if hit_keyword is not None and hit_score >= threshold and min_frames <= duration <= max_frames:
            detections.append((hit_keyword, hit_score, start, end))
            cur_hyps = [(tuple(), (1.0, 0.0, []))]
            hit_keyword, hit_score = None, 1.0
    lines = ['{} detected {} {:.3f}\n'.format(key, w, s) for w, s, _, _ in detections]
    return (lines or ['{} rejected\n'.format(key)]), detections            # :375-376


def stream_score_text(keys, probs, lengths, keywords_token, **kw):
    """The score file of a batch: probs (B, T, V), lengths (B,)."""
    out = []
    for b, key in enumerate(keys):
        out.extend(stream_score(key, probs[b, :int(lengths[b])], keywords_token, **kw)[0])
    return ''.join(out)


def split_mixed_label(input_str):
    """compute_det_ctc.py:30-41."""
    tokens = []
    s = input_str.lower()
    while len(s) > 0:
        match = re.match(r"[A-Za-z!?,<>()']+", s)
        word = match.group(0) if match is not None else s[0:1]
        tokens.append(word)
        s = s.replace(word, '', 1).strip(' ')
    return tokens


def space_mixed_label(input_str):
    """compute_det_ctc.py:44-47."""
    return ''.join(f'{sub} ' for sub in split_mixed_label(input_str)).strip()


def load_label_and_score(keywords_list, label_list, score_lines, true_keywords):
    """compute_det_ctc.py:50-124 with the files already read (label objects, score lines)."""
    score_table = {}
    for line in score_lines:
        arr = line.strip().split()
        key = arr[0]
        if arr[1] == 'detected':
            keyword = true_keywords[arr[2]]
            if key not in score_table:
                score_table[key] = {'kw': space_mixed_label(keyword), 'confi': float(arr[3])}
        elif key not in score_table:
            score_table[key] = {'kw': 'unknown', 'confi': -1.0}
    table = {}
    for keyword in keywords_list:
        keyword = space_mixed_label(true_keywords[keyword])
        table[keyword] = {'keyword_table': {}, 'keyword_duration': 0.0, 'filler_table': {}, 'filler_duration': 0.0}
    for obj in label_list:
        key, duration = obj['key'], obj['duration']
        txt_lr = ' ' + space_mixed_label(obj['txt']) + ' '
        assert key in score_table
        for keyword in keywords_list:
            keyword = space_mixed_label(true_keywords[keyword])
            side = 'keyword' if txt_lr.find(' ' + keyword + ' ') != -1 else 'filler'
            if keyword == score_table[key]['kw']:
                table[keyword][side + '_table'].update({key: score_table[key]['confi']})
            else:
                table[keyword][side + '_table'].update({key: -1.0})
            table[keyword][side + '_duration'] += duration
    return table


def det_stats_text(label_list, score_lines, true_keywords, step=0.01):
    """compute_det_ctc.py:228-281 -> {stats file name: text}."""
    keywords_list = list(true_keywords)
    table = load_label_and_score(keywords_list, label_list, score_lines, true_keywords)
    out = {}
    for keyword in keywords_list:
        keyword = space_mixed_label(true_keywords[keyword])
        keyword_num = len(table[keyword]['keyword_table'])
        filler_dur = table[keyword]['filler_duration']
        filler_num = len(table[keyword]['filler_table'])
        assert keyword_num > 0 and filler_num > 0
        rows = []
        threshold = 0.0
        while threshold <= 1.0:
            num_false_reject = sum(1 for c in table[keyword]['keyword_table'].values() if c < threshold)
            num_false_alarm = sum(1 for c in table[keyword]['filler_table'].values() if c >= threshold)
            num_false_alarm = max(num_false_alarm, 1e-6)
            rows.append('{:.3f} {:.6f} {:.6f}\n'.format(threshold, num_false_alarm / (filler_dur / 3600.0),
                                                        num_false_reject / keyword_num))
            threshold += step
        out['stats.' + keyword.replace(' ', '_') + '.txt'] = ''.join(rows)
    return out


PLANT_V = 48
PLANTS = [[5, 9, 23], [31, 7, 23, 23], [23, 23], [40, 12], [5, 9, 40], [17, 23], [31, 7]]   # 40, 12, 17: no keyword


def plant_logits(B, T, seed):
    """(B, T, V) logits: blank-dominated rows with token sequences planted (keyword ones, partial ones and ones of
    non-keyword tokens, whose rows the filter empties), each token held 1-4 rows at its own sharpness, so hit scores
    fall on both sides of the thresholds; now and then a competitor above the 0.05 gate."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(B, T, PLANT_V, generator=g) * 0.3
    for b in range(B):
        logits[b, :, 0] += 7.0
        t = int(torch.randint(1, 8, (1,), generator=g))
        while t < T:
            seq = PLANTS[int(torch.randint(0, len(PLANTS), (1,), generator=g))]
            for tok in seq:
                sharp = -1.0 + 7.0 * float(torch.rand(1, generator=g))
                for _ in range(int(torch.randint(1, 5, (1,), generator=g))):
                    if t < T:
                        logits[b, t, tok] += sharp + 7.0
                        if torch.rand(1, generator=g) < 0.2:
                            logits[b, t, int(torch.randint(0, PLANT_V, (1,), generator=g))] += sharp + 4.5
                        t += 1
                t += int(torch.randint(0, 3, (1,), generator=g))
            t += int(torch.randint(2, 20, (1,), generator=g))
    return logits
