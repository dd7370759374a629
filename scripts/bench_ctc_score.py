#!/usr/bin/env python
"""CTC test-set scoring throughput (stage 3 of the CTC recipes): fsmn_ctc at the shipped size (80 mel x context (2, 2)
= 400 inputs, 2599 outputs, frame_skip 3) over a synthetic test set of utterances of 1-8 s.  Per batch size: the device
time of the model (Fbank + context expansion + forward_softmax) and of the stream-score decode (ctc_stream_score, one
launch) from CUDA events, utterances/s and audio-hours/s of the two together; the DET statistics at step 0.001 over
the test set's score file (compute_det_ctc end to end, and the device sweep alone); the CPU oracle of
stream_score_ctc.py on a subset.  A randomly initialised model never puts a token above the 0.05 gate, so the decode
runs on CTC-like posteriors of the same shape instead (blank-dominated rows with keyword and filler token sequences
planted, oracle/ctc_score_oracle.py plant_logits; the other 2551 outputs are background): the decode's cost depends on how
often the beam moves.  The GPU's name, power limit and max SM clock are read in the same run.  Prints one JSON line.

    python scripts/bench_ctc_score.py [--utterances 8192] [--batches 256 4096] [--oracle-utterances 16] [--out FILE]
"""
import argparse
import io
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ctc_score_oracle as SO                                                     # noqa: E402
from oracle.ctc_score_oracle import plant_logits                                         # noqa: E402
from wekws_b200 import (Fbank, compute_det_ctc, context_expansion, ctc_det_sweep, ctc_stream_score,  # noqa: E402
                        det_thresholds, init_model, model_config, synth, write_ctc_stream_scores)

KEYWORDS = {"hi_xiaowen": {"token_id": [5, 9, 23]}, "nihao_wenwen": {"token_id": [31, 7, 23, 23]}}
SKIP, CTX, V = 3, (2, 2), 2599


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": int(clock)}


def planted_probs(planted, idx, T):
    """(len(idx), T, V) posteriors: utterance i gets planted[i % 128] (the planting loop is slow Python) in the first 48
    outputs, background after."""
    logits = torch.randn(len(idx), T, V, device="cuda") * 0.3
    logits[:, :, :planted.size(2)] = planted[idx % planted.size(0), :T].cuda()
    return logits.softmax(2)


def frame_counts(n):
    """Fbank frames of each utterance (25 ms windows, 10 ms hop), computed on the host outside the timed window."""
    return torch.tensor([max(0, (int(v) - 400) // 160 + 1) for v in n], dtype=torch.int32)


def features(fb, pcm, flen):
    return context_expansion(fb(pcm), CTX[0], CTX[1], SKIP, lengths=flen)


def batch_pcm(base, n_all, idx):
    """Utterance i is the first n_all[i] samples of base[i % 64]."""
    n = n_all[idx]
    return base[idx % base.size(0), :int(n.max())].cuda(), n


def bench_batch(model, fb, base, n_all, planted, B, reps):
    model_ms, dec_ms, sc = [], [], None
    for r in range(reps):
        idx = torch.arange(r * B, (r + 1) * B) % n_all.numel()
        pcm, n = batch_pcm(base, n_all, idx)
        flen = frame_counts(n)
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        x, lens = features(fb, pcm, flen)
        with torch.no_grad():
            probs, _ = model.forward_softmax(x)
        e1.record()
        probs = planted_probs(planted, idx, probs.size(1))
        e2.record()
        sc = ctc_stream_score(probs, lens, KEYWORDS, frame_skip=SKIP)
        e3.record()
        torch.cuda.synchronize()
        model_ms.append(e0.elapsed_time(e1))
        dec_ms.append(e2.elapsed_time(e3))
    return model_ms, dec_ms, sc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utterances", type=int, default=8192)
    ap.add_argument("--batches", type=int, nargs="+", default=[256, 4096])
    ap.add_argument("--oracle-utterances", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator().manual_seed(0)
    N = a.utterances
    n_all = torch.randint(16000, 8 * 16000 + 1, (N,), generator=g)
    base = synth.pcm_int16(64, 8 * 16000, seed=1)
    model = synth.randomize_(init_model(model_config("fsmn", input_dim=400, output_dim=V)), seed=11).eval().cuda()
    fb = Fbank(80)
    rows = (n_all - 400) // 160 + 1                                         # Fbank frames, then context + skip
    planted = plant_logits(128, int(((rows.max() - CTX[1] + SKIP - 1) // SKIP)), 5)
    line = {"workload": "ctc_stream_score_fsmn_ctc_testset", **gpu_info(), "utterances": N,
            "audio_hours": round(float(n_all.sum()) / 16000 / 3600, 3), "results": []}

    keys = [f"utt{i:06d}" for i in range(N)]
    score_text = io.StringIO()
    for B in a.batches:
        reps = max(1, N // B)
        bench_batch(model, fb, base, n_all, planted, B, 1)                # warm-up: every shape of this batch size
        model_ms, dec_ms, sc = bench_batch(model, fb, base, n_all, planted, B, reps)
        tot = np.array(model_ms) + np.array(dec_ms)
        audio_s = float(n_all[torch.arange(reps * B) % N].sum()) / 16000
        line["results"].append({
            "batch": B, "batches_timed": reps,
            "model_ms_per_batch_median": round(float(np.median(model_ms)), 3),
            "decode_ms_per_batch_median": round(float(np.median(dec_ms)), 3),
            "utterances_per_s": round(reps * B / (tot.sum() / 1e3), 1),
            "audio_hours_per_s": round(audio_s / 3600 / (tot.sum() / 1e3), 4),
            "detections_last_batch": int(sc.count.sum())})
    # the score file of the whole test set (batches of the largest size), then DET at step 0.001
    B = max(a.batches)
    labels, unexact = [], 0
    for s in range(0, N, B):
        idx = torch.arange(s, min(N, s + B))
        pcm, n = batch_pcm(base, n_all, idx)
        x, lens = features(fb, pcm, frame_counts(n))
        probs = planted_probs(planted, idx, x.size(1))
        sc = ctc_stream_score(probs, lens, KEYWORDS, frame_skip=SKIP)
        # utterances the writer would refuse (decoder overflow, > max_detections) are written as rejected and counted
        bad = (sc.overflow != 0) | (sc.count > sc.max_detections)
        unexact += int(bad.sum())
        sc.count[bad] = 0
        sc.overflow[bad] = 0
        write_ctc_stream_scores(score_text, keys[s:s + len(idx)], sc)
        if s == 0:
            sub = (probs[:a.oracle_utterances].cpu(), lens[:a.oracle_utterances])
    rng = np.random.default_rng(0)
    for i in range(N):
        labels.append({"key": keys[i], "txt": "hi_xiaowen" if rng.random() < 0.3 else "nihao_wenwen" if
                       rng.random() < 0.3 else "filler", "duration": float(n_all[i]) / 16000})
    lines = score_text.getvalue().splitlines(True)
    true_kw = {"hi_xiaowen": "hi_xiaowen", "nihao_wenwen": "nihao_wenwen"}
    compute_det_ctc(labels, lines, true_kw, 0.001)                        # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    compute_det_ctc(labels, lines, true_kw, 0.001)
    det_wall = time.perf_counter() - t0
    thr = det_thresholds(0.001).cuda()
    ck = torch.rand(N // 3, dtype=torch.float64, device="cuda")
    cf = torch.rand(N - N // 3, dtype=torch.float64, device="cuda")
    ctc_det_sweep(ck, cf, thr)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        ctc_det_sweep(ck, cf, thr)
    e1.record()
    torch.cuda.synchronize()
    line["score_file"] = {"lines": len(lines), "detected": sum(" detected " in x for x in lines),
                          "utterances_not_exact": unexact}
    line["det_step_0.001"] = {"keywords": 2, "thresholds": int(thr.numel()),
                              "compute_det_ctc_wall_ms": round(det_wall * 1e3, 3),
                              "sweep_kernel_ms_per_keyword": round(e0.elapsed_time(e1) / 20, 4)}
    # CPU comparison: the oracle of stream_score_ctc.py's decode loop on a subset (same probabilities)
    p, ln = sub
    t0 = time.perf_counter()
    for b in range(p.size(0)):
        SO.stream_score(keys[b], p[b, :int(ln[b])], KEYWORDS, frame_skip=SKIP)
    cpu = time.perf_counter() - t0
    line["cpu_oracle_decode"] = {"utterances": int(p.size(0)), "utterances_per_s": round(p.size(0) / cpu, 3),
                                 "audio_hours_per_s": round(float(n_all[:p.size(0)].sum()) / 16000 / 3600 / cpu, 6)}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
