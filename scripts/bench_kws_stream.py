#!/usr/bin/env python
"""Streaming CTC keyword spotter throughput (wekws_b200.KeyWordSpotter): 0.3 s int16 chunks per stream per call (the
interval of the reference demo, wekws/bin/stream_kws_ctc.py:558-560) for fsmn_ctc (80 mel, context (2, 2), skip 3) and
ds_tcn_ctc (40 mel, no context), both with 2599 outputs, at several stream counts.  Per configuration: audio-hours/s
over a timed region of >= --seconds, p50 / p99 latency of one forward() (results on the host), the device time of each
stage from CUDA events in a separate pass, and kernel launches per call.  Also the CPU baseline (the oracle spotter,
one stream) and the GPU's name, power limit and max SM clock read in the same run.  Prints one JSON line.

    python scripts/bench_kws_stream.py [--streams 1 256 1024 4096] [--seconds 1.0] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import kws_oracle as O                      # noqa: E402
from oracle import kws_stream_oracle as KO              # noqa: E402
from wekws_b200 import KeyWordSpotter, _native, init_model, model_config, synth   # noqa: E402

CHUNK = int(0.3 * 16000)
KEYWORDS = {"hi_xiaowen": {"token_id": [5, 9, 17, 23]}, "nihao_wenwen": {"token_id": [31, 7, 23, 23]}}
MODELS = {
    "fsmn_ctc": dict(cfg=lambda: model_config("fsmn", input_dim=400, output_dim=2599), mel=80, context=(2, 2), skip=3),
    "ds_tcn_ctc": dict(cfg=lambda: model_config("ds_tcn", input_dim=40, output_dim=2599, activation="identity"),
                       mel=40, context=None, skip=1),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().split(",")]
    return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": int(clock)}


def run(name, B, seconds, warmup):
    m = MODELS[name]
    model = synth.randomize_(init_model(m["cfg"]())).eval().cuda()
    sp = KeyWordSpotter(model, KEYWORDS, 0.5, B, "cuda", num_mel_bins=m["mel"], context=m["context"],
                        frame_skip=m["skip"])
    pcm = synth.pcm_int16(min(B, 64), CHUNK * 8, seed=1).cuda()
    chunks = [pcm[torch.arange(B) % pcm.size(0), i * CHUNK:(i + 1) * CHUNK].contiguous() for i in range(8)]
    for i in range(warmup):
        sp.forward(chunks[i % 8])
    torch.cuda.synchronize()
    lat, calls, t0 = [], 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        t = time.perf_counter()
        sp.forward(chunks[calls % 8])
        lat.append(time.perf_counter() - t)
        calls += 1
    wall = time.perf_counter() - t0
    # launches of one call, then the per-stage device time (CUDA events at the stage boundaries, a separate pass)
    n0 = _native.launch_count()
    sp.forward(chunks[0])
    launches = _native.launch_count() - n0
    stages, evs = {}, []
    sp.stage_hook = lambda s: evs.append((s, torch.cuda.Event(enable_timing=True))) or evs[-1][1].record()
    reps = max(3, min(50, calls))
    for i in range(reps):
        evs.clear()
        sp.forward(chunks[i % 8])
        for (s, a), (_, b) in zip(evs[:-1], evs[1:]):
            stages[s] = stages.get(s, 0.0) + a.elapsed_time(b) / reps
    sp.stage_hook = None
    return {"model": name, "streams": B, "calls": calls,
            "audio_hours_per_s": round(B * 0.3 * calls / wall / 3600, 3),
            "latency_ms_p50": round(1e3 * float(np.percentile(lat, 50)), 3),
            "latency_ms_p99": round(1e3 * float(np.percentile(lat, 99)), 3),
            "stage_ms": {k: round(v, 4) for k, v in stages.items()}, "launches_per_call": launches}


def cpu_baseline(name, seconds):
    m = MODELS[name]
    cfg = m["cfg"]()
    model = synth.randomize_(init_model(cfg)).eval()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    k = KO.KeyWordSpotter(KEYWORDS, 0.5, lambda f, c: O.kws_forward(sd, cfg, f, c), num_mel_bins=m["mel"],
                          context=m["context"], frame_skip=m["skip"])
    pcm = synth.pcm_int16(1, CHUNK * 8, seed=1)[0].numpy()
    k.forward(pcm[:CHUNK])
    calls, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        k.forward(pcm[(calls % 8) * CHUNK:(calls % 8 + 1) * CHUNK])
        calls += 1
    return {"model": name, "streams": 1, "audio_hours_per_s": round(0.3 * calls / (time.perf_counter() - t0) / 3600, 6)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", type=int, nargs="+", default=[1, 256, 1024, 4096])
    ap.add_argument("--models", nargs="+", default=list(MODELS))
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.backends.cuda.matmul.allow_tf32 = False
    line = {"workload": "kws_stream_0.3s_chunks", **gpu_info(),
            "results": [run(n, B, a.seconds, a.warmup) for n in a.models for B in a.streams],
            "cpu_baseline_oracle": [cpu_baseline(n, a.seconds) for n in a.models]}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
