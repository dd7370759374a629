#!/usr/bin/env python
"""Benchmark of the WeKws streaming KWS forward path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--no-extras]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1]): the `mdtc` model (hidden 64, 1+4x4 DS-dilated blocks, k=5),
80-dim features, B = 1024 concurrent streams per GPU, chunk T = 40 frames, streaming caches (B,64,244)
carried from step to step.  A "step" is one pass of KWSModel.forward over one batch of B x T synthetic
frames.  Metric: audio-hours/sec = frames/sec / 360000 (100 frames per second).

* `value`      whole-job throughput of EXACTLY --steps steps after --warmup warm-ups, inputs resident in HBM,
               device-timed (CUDA events) between barriers, max over ranks.
* `e2e`        same metric through the public Python surface (wekws_b200.KWSModel.forward) with the step's
               features coming from pinned HOST memory (H2D) and its posteriors read back (D2H) inside the
               timed region; the streaming cache stays on the device as it does in the reference's own
               streaming loop (stream_kws_ctc.py:487).  The e2e loop has its own length (`e2e.steps`): it
               warms up until the per-step time is stable (>= 0.5 s) and then times >= 1 s, the same number of
               steps on every rank, so a 20-step driver run does not time cold PCIe / first-touch effects.
               Each rank binds itself (and therefore its pinned buffers, first touch) to the CPUs local to
               its GPU before anything is allocated.
* `roofline`   dominant kernel (mdtc_tc_kernel for the headline workload): algorithmic bytes per launch
               (idim*4 + odim*4 + 2*cache_bytes_per_stream/T = 3447 B/frame, SURVEY 8d) / mean launch
               duration measured with CUDA events, against the measured HBM copy bandwidth in
               MEASURED_PEAKS.json; plus the bf16 tensor-pipe figure for the tcgen05 kernels.
* `cpu_baseline` / `--impl reference`: the oracle port of the reference's PyTorch CPU path
               (oracle/kws_oracle.py, same ATen ops) on the host cores, run in a fresh process with the
               full CPU affinity; thread count and sub-batch chosen by the median of 5 timed calls each.
* `extra_workloads`: BASELINE configs[2..4] per GPU -- GRU B=512 T=1, tcn and ds_tcn B=1024 T=40, raw
               PCM -> posterior 1250 x 1 s clips (p50 / p99 batch latency) -- each with its own value, e2e,
               roofline and clock record, inside a bounded time budget.
Multi-GPU: streams are independent -> each rank owns its own B streams ("weak" scaling), no collective
on the data path; torch.distributed (NCCL) is used only for the barrier and the max-over-ranks time.
Between timed steps the working set rotates over NSETS independent stream sets (> 126 MB L2).
--dump-outputs DIR: what the last timed step of the headline workload returned to its caller, written after the timed
               loop as DIR/posteriors.npy (B, T, odim) and DIR/cache.npy (the streaming cache), float32, rank 0.  At
               most DUMP_BYTES in all: an array that does not fit keeps a fixed, seeded sample of its streams.  Inputs
               and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FRAMES_PER_HOUR = 360000.0
WORKLOADS = {
    # name: (model, B per GPU, T, idim)
    "mdtc_b1024_t40": ("mdtc", 1024, 40, 80),
    "gru_b512_t1": ("gru", 512, 1, 80),
    "tcn_b1024_t40": ("tcn", 1024, 40, 80),
    "ds_tcn_b1024_t40": ("ds_tcn", 1024, 40, 80),
    # BASELINE configs[4]: raw PCM -> posterior, 10 000 one-second clips over 8 GPUs = 1250 clips per GPU;
    # T = 98 frames per clip (16000 samples), every clip starts a stream (no cache carried)
    "pcm_e2e_1250x1s": ("mdtc", 1250, 98, 80),
}
EXTRAS = ["gru_b512_t1", "tcn_b1024_t40", "ds_tcn_b1024_t40", "pcm_e2e_1250x1s"]
PCM_SAMPLES = 16000
NSETS = 4
DUMP_BYTES = 64 * 10 ** 6
METRIC = "audio-hours/sec KWS scoring (frames/sec / 360000)"
DTYPE = "f32 I/O, bf16x3 tensor GEMMs (fp32 accumulate, ~2^-17; GRU and front-end: fp32 FMA)"


# ------------------------------------------------------------------------------------------- host placement
def bind_to_gpu_cpus(local_gpu):
    """Pins this process to the CPUs local to its GPU (NUMA node of the PCIe root) BEFORE torch / CUDA allocate
    anything, so the pinned staging buffers are first-touched on that node.  Returns (description, original
    affinity) -- the CPU baseline runs in a child with the original affinity."""
    try:
        orig = os.sched_getaffinity(0)
    except Exception:
        return "affinity unavailable", None
    try:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = local_gpu
        if vis:
            parts = [p.strip() for p in vis.split(",") if p.strip()]
            if local_gpu < len(parts) and parts[local_gpu].isdigit():
                idx = int(parts[local_gpu])
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        words = (max(orig) // 64) + 1 if orig else 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i * 64 + b for i, w in enumerate(mask) for b in range(64) if (int(w) >> b) & 1} & orig
        if cpus and cpus != orig:
            os.sched_setaffinity(0, cpus)
            lo, hi = min(cpus), max(cpus)
            return f"bound to the {len(cpus)} CPUs local to GPU {idx} (cpu {lo}..{hi})", orig
        return "GPU-local CPU set == process CPU set (single NUMA domain)", orig
    except Exception as e:  # no NVML / no permission: keep going unbound
        return f"not bound ({type(e).__name__})", orig


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return {}, 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes_per_frame(model, T, idim, odim=1):
    """SURVEY 8d: features in + posteriors out + streaming cache read once and written once."""
    cache_bytes = {"mdtc": 64 * 244 * 4, "mdtc_small": 32 * 184 * 4, "ds_tcn": 256 * 105 * 4,
                   "tcn": 64 * 105 * 4, "gru": 2 * 128 * 4}[model]
    return idim * 4 + odim * 4 + 2.0 * cache_bytes / T


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed regions (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------- CPU reference arm
def build_oracle_model(model_name, idim):
    import torch
    from wekws_b200 import init_model, model_config, synth
    cfg = model_config(model_name, input_dim=idim)
    torch.manual_seed(777)
    m = synth.randomize_(init_model(cfg), seed=777).eval()
    return cfg, m


def cpu_reference_run(workload, steps, warmup, budget_s):
    """The reference's CPU PyTorch path (oracle port, same ATen ops) on the host cores.  One step = the workload's
    full per-GPU batch (B streams x T frames; raw-PCM workloads: per-clip kaldi-style Fbank + forward, the way the
    reference does it), executed as ceil(B / sub) sub-batches; (threads, sub) = best median of 5 timed calls.
    Runs `warmup` untimed and up to `steps` timed steps, stopping early (>= 3 steps) when budget_s is spent."""
    import torch
    from oracle import kws_oracle as O
    from wekws_b200 import synth
    model_name, B, T, idim = WORKLOADS[workload]
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cfg, m = build_oracle_model(model_name, idim)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    gru = cfg["backbone"]["type"] == "gru"
    pcm_mode = workload.startswith("pcm_")
    if pcm_mode:
        pcm = synth.pcm_int16(B, PCM_SAMPLES, seed=1234).float()
    else:
        x = synth.features(B, T, idim, seed=4321)

    def make_step(sub):
        slices = [(s, min(B, s + sub)) for s in range(0, B, sub)]
        caches = [torch.zeros(cfg["backbone"]["num_layers"], e - s, cfg["hidden_dim"]) if gru else None
                  for s, e in slices]

        def step():
            for i, (s, e) in enumerate(slices):
                if pcm_mode:      # per-clip Fbank (kaldi.fbank is single-waveform, kaldi.py:135-137), batched forward
                    f = torch.stack([O.fbank(pcm[b]) for b in range(s, e)])
                    O.kws_forward(sd, cfg, f, None)
                else:
                    _, caches[i] = O.kws_forward(sd, cfg, x[s:e], caches[i])
        return step

    def median_time(fn, n):
        fn()
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return statistics.median(ts)

    # probe on a slice of the batch: threads x sub-batch, median of 5 timed calls each, bounded in time
    threads = [n for n in dict.fromkeys((16, 32, 8, 64, 4, ncpu, 1)) if n <= ncpu]   # likely winners first (time-bounded)
    subs = sorted({s for s in (64, 256, B) if s <= B}) if not pcm_mode else [min(B, 125)]
    best = None
    t_probe = time.perf_counter()
    for sub in subs:
        probe_b = min(B, sub)
        xs = None if pcm_mode else x[:probe_b]
        for n in threads:
            torch.set_num_threads(n)
            c0 = [torch.zeros(cfg["backbone"]["num_layers"], probe_b, cfg["hidden_dim"]) if gru else None]

            def call():
                if pcm_mode:
                    f = torch.stack([O.fbank(pcm[b]) for b in range(probe_b)])
                    O.kws_forward(sd, cfg, f, None)
                else:
                    _, c0[0] = O.kws_forward(sd, cfg, xs, c0[0])
            dt = median_time(call, 5) / probe_b           # seconds per stream-chunk
            if best is None or dt < best[0]:
                best = (dt, n, sub)
            if time.perf_counter() - t_probe > 0.45 * budget_s:
                break
    _, cores, sub = best
    torch.set_num_threads(cores)
    step = make_step(sub)
    for _ in range(warmup):
        step()
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and len(times) >= 3:
            break
    total = sum(times)
    fps = B * T * len(times) / total
    return {"value": fps / FRAMES_PER_HOUR, "unit": "audio-hours/s", "cores": cores, "kind": "port",
            "frames_per_sec": fps, "ms_per_step": 1e3 * total / len(times), "steps": len(times), "warmup": warmup,
            "sample": f"oracle port (torch CPU) of {workload}: {len(times)} steps of the full per-GPU batch "
                      f"({B} x {T} frames, as sub-batches of {sub}), state carried; threads/sub-batch = best median "
                      f"of 5 calls over {threads} x {subs} -> {cores} threads; host exposes {ncpu} CPUs"}


def reference_line(args, config, r):
    return {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": "audio-hours/s", "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": r["warmup"], "ms_per_step": r["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "frames_per_sec": r["frames_per_sec"],
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": r["value"], "unit": "audio-hours/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


def workload_config(workload, gpus):
    model_name, B, T, idim = WORKLOADS[workload]
    cfg = {"workload": f"{model_name}: {B} streams/GPU x {T}-frame chunks, {idim}-dim features, cache carried",
           "model_cfg": model_name, "streams_per_gpu": B, "chunk_frames": T, "feature_dim": idim,
           "global_streams": B * max(gpus, 1), "parallelism": f"streams sharded x{max(gpus, 1)} (no collective)",
           "l2": f"working set rotates over {NSETS} independent stream sets (> 126 MB L2 for the conv models)"}
    if workload.startswith("pcm_"):
        cfg["workload"] = (f"raw int16 PCM -> Fbank -> {model_name}: {B} one-second clips/GPU "
                           f"({T} frames each), start of stream")
    return cfg


# ------------------------------------------------------------------------------------------- our arm
def dump_outputs(out_dir, arrays):
    """arrays: name -> (tensor, index of its stream dimension), written in this order as out_dir/<name>.npy (float32).
    An array larger than what is left of DUMP_BYTES keeps the streams torch.randperm(n, generator seeded with 0)[:k],
    in ascending order, for the largest k that fits."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for name, (t, dim) in arrays.items():
        a = t.detach().float().cpu()
        n = a.shape[dim]
        k = min(n, left // (4 * a.numel() // n))
        if k < n:
            keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:k].sort().values
            a = a.index_select(dim, keep)
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())
        left -= 4 * a.numel()


class Runner:
    def __init__(self, dev, rank, world, dist):
        self.dev, self.rank, self.world, self.dist = dev, rank, world, dist

    def barrier(self):
        import torch
        torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def reduce(self, v, op="max"):
        import torch
        t = torch.tensor([float(v)], device=self.dev, dtype=torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def run(self, workload, steps, warmup, min_region_s=0.0, dump_dir=None):
        """value / latency / e2e / roofline of one workload.  steps, warmup: the device-resident timed loop (exactly
        as given when min_region_s == 0; extras pass min_region_s to size the loop by time instead).  dump_dir: where
        dump_outputs() writes what the last timed step returned."""
        import torch
        from wekws_b200 import _native, init_model, model_config, synth
        dev, rank, world = self.dev, self.rank, self.world
        model_name, B, T, idim = WORKLOADS[workload]
        cfg = model_config(model_name, input_dim=idim)
        torch.manual_seed(777)
        model = synth.randomize_(init_model(cfg), seed=777).eval().to(dev)
        gru = model_name == "gru"
        cshape = (2, B, 128) if gru else (B, model.hdim, model.backbone.padding)
        pcm_mode = workload.startswith("pcm_")
        if pcm_mode:
            from wekws_b200 import Fbank, Pipeline
            fb = Fbank(idim)
            pipe = Pipeline(fb, model)
            pcm = [synth.pcm_int16(B, PCM_SAMPLES, seed=1234 + rank * 17 + s).to(dev) for s in range(NSETS)]
            feat_buf = torch.empty(B, T, idim, device=dev)
            feats = [feat_buf] * NSETS
            caches = [None] * NSETS
        else:
            feats = [synth.features(B, T, idim, seed=4321 + rank * 17 + s).to(dev) for s in range(NSETS)]
            caches = [torch.zeros(cshape, device=dev) for _ in range(NSETS)]

        last = [None]          # (posteriors, cache) the latest step returned

        def step(i):
            s = i % NSETS
            if pcm_mode:
                last[0] = pipe(pcm[s])
            else:
                y, caches[s] = model(feats[s], caches[s])
                last[0] = (y, caches[s])

        # ---------------- device-resident throughput (`value`) ------------------------------------------------
        for i in range(max(warmup, 3)):
            step(i)
        self.barrier()
        if min_region_s > 0:          # extras: size the loop by time (same count on every rank)
            t0 = time.perf_counter()
            for i in range(20):
                step(i)
            torch.cuda.synchronize()
            per = (time.perf_counter() - t0) / 20
            steps = int(self.reduce(max(20, min(20000, math.ceil(min_region_s / max(per, 1e-6))))))
            self.barrier()
        sampler = ClockSampler(dev.index).start() if rank == 0 else None
        n0 = _native.launch_count()
        t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin.record()
        for i in range(steps):
            step(i)
        t_end.record()
        self.barrier()
        launches = _native.launch_count() - n0
        if dump_dir is not None and rank == 0:
            dump_outputs(dump_dir, {"posteriors": (last[0][0], 0), "cache": (last[0][1], 1 if gru else 0)})
        total_ms = self.reduce(t_begin.elapsed_time(t_end))
        fps = B * T * steps * world / (total_ms * 1e-3)
        # per-launch durations (roofline, p50/p99) from a separate pass: bracketing every step with events costs
        # more host time than a 10 us kernel takes, so it stays out of the timed region
        nlat = 200
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nlat)]
        for i in range(nlat):
            ev[i][0].record()
            step(i)
            ev[i][1].record()
        self.barrier()
        per_launch_ms = [a.elapsed_time(b) for a, b in ev]

        # ---------------- end to end through the public API with host buffers (`e2e`) --------------------------
        src = pcm if pcm_mode else feats
        h_in = [t.cpu().pin_memory() for t in src]
        h_out = [torch.empty(B, T, model.odim).pin_memory() for _ in range(2)]
        d_in = [torch.empty_like(src[0]) for _ in range(2)]
        copy_stream, main_stream = torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
        in_ready = [torch.cuda.Event() for _ in range(2)]
        in_free = [torch.cuda.Event() for _ in range(2)]

        def e2e_run(nsteps):
            # H2D of step i+1 overlaps the kernel of step i (separate copy stream, double buffered);
            # every step's posteriors are copied back to pinned host memory
            with torch.cuda.stream(copy_stream):
                d_in[0].copy_(h_in[0], non_blocking=True)
                in_ready[0].record(copy_stream)
            for i in range(nsteps):
                b, s = i & 1, i % NSETS
                if i + 1 < nsteps:
                    nb = (i + 1) & 1
                    with torch.cuda.stream(copy_stream):
                        if i >= 1:
                            copy_stream.wait_event(in_free[nb])
                        d_in[nb].copy_(h_in[(i + 1) % NSETS], non_blocking=True)
                        in_ready[nb].record(copy_stream)
                main_stream.wait_event(in_ready[b])
                if pcm_mode:
                    y, _ = pipe(d_in[b])
                else:
                    y, caches[s] = model(d_in[b], caches[s])
                in_free[b].record(main_stream)
                h_out[b].copy_(y, non_blocking=True)
            main_stream.synchronize()

        def e2e_timed(n):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            e2e_run(n)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        # warm-up until the per-step time is stable (two consecutive ~0.1 s chunks within 5 %) and >= 0.5 s have
        # passed (at most 3 s): first-touch of the pinned buffers, PCIe link power state, clocks
        per, t_w = e2e_timed(8), time.perf_counter()
        while True:
            n = max(8, min(4000, int(100.0 / max(per, 1e-3))))
            new = e2e_timed(n)
            stable = abs(new - per) <= 0.05 * per
            per = new
            el = time.perf_counter() - t_w
            if (stable and el >= 0.5) or el >= 3.0:
                break
        e2e_steps = int(self.reduce(max(16, min(40000, math.ceil(1000.0 / max(per, 1e-3))))))
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        e2e_run(e2e_steps)
        e1.record()
        self.barrier()
        e2e_ms = self.reduce(e0.elapsed_time(e1))
        e2e_fps = B * T * e2e_steps * world / (e2e_ms * 1e-3)
        # serialized per-batch completion latency through the host API (H2D -> kernels -> D2H, one batch in flight)
        e2e_lat = None
        if pcm_mode or gru:
            ls = []
            for i in range(100):
                a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                d_in[0].copy_(h_in[i % NSETS], non_blocking=True)
                if pcm_mode:
                    y, _ = pipe(d_in[0])
                else:
                    y, caches[0] = model(d_in[0], caches[0])
                h_out[0].copy_(y, non_blocking=True)
                b2.record()
                torch.cuda.synchronize()
                ls.append(a.elapsed_time(b2))
            ls.sort()
            e2e_lat = {"p50_ms": ls[len(ls) // 2], "p99_ms": ls[min(len(ls) - 1, int(0.99 * len(ls)))],
                       "what": "one batch in flight: pinned H2D + kernels + D2H of the posteriors"}
        clocks = sampler.stop() if sampler is not None else None

        # ---------------- single-stream chunk latency (BASELINE configs[0] shape on the GPU) -------------------
        lat = None
        if rank == 0 and not pcm_mode:
            x1 = synth.features(1, T, idim, seed=1).to(dev)
            c1 = torch.zeros((2, 1, 128) if gru else (1, model.hdim, model.backbone.padding), device=dev)
            for _ in range(20):
                _, c1 = model(x1, c1)
            torch.cuda.synchronize()
            ls = []
            for _ in range(200):
                a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                _, c1 = model(x1, c1)
                b2.record()
                torch.cuda.synchronize()
                ls.append(a.elapsed_time(b2))
            lat = statistics.median(ls)
        if rank != 0:
            return None

        peaks, peak, peak_src = measured_peaks()
        bpf = algorithmic_bytes_per_frame(model_name, T, idim, model.odim)
        if pcm_mode:   # PCM in + posteriors out + the new cache written once (no cache read at start of stream)
            bpf = PCM_SAMPLES * 2.0 / T + model.odim * 4 + (64 * 244 * 4) / T
        launch_ms = statistics.mean(per_launch_ms)
        srt = sorted(per_launch_ms)
        p99_ms = srt[min(len(srt) - 1, int(0.99 * len(srt)))]
        achieved = bpf * B * T / (launch_ms * 1e-3) / 1e9
        traffic = None
        prof = os.path.join(ROOT, "profiles", "dominant_kernel.json")
        if os.path.exists(prof):
            try:
                with open(prof) as f:
                    traffic = json.load(f).get(workload, {}).get("dram_bytes_per_launch")
            except Exception:
                traffic = None
        tc = bool(model.uses_tensor_cores(T, B))
        kname = ("gru_tc_kernel" if tc else "gru_kernel") if gru else ({"tcn": "tcn_tc_kernel", "ds_tcn": "dstcn_tc_kernel"}.get(
            model_name, "mdtc_tc_kernel") if tc else "conv_backbone_kernel")
        flop_per_frame = {"mdtc": 299776, "tcn": 272512, "ds_tcn": 582144, "gru": 413952}.get(model_name)
        res = {
            "workload": workload, "config": workload_config(workload, world),
            "value": fps / FRAMES_PER_HOUR, "unit": "audio-hours/s", "frames_per_sec": fps, "steps": steps,
            "ms_per_step": total_ms / steps,
            "p50_step_latency_ms": statistics.median(per_launch_ms), "p99_step_latency_ms": p99_ms,
            "p50_chunk_latency_ms_1stream": lat, "clocks": clocks,
            "e2e": {"value": e2e_fps / FRAMES_PER_HOUR, "unit": "audio-hours/s", "frames_per_sec": e2e_fps,
                    "h2d_bytes_per_step": (B * PCM_SAMPLES * 2) if pcm_mode else (B * T * idim * 4),
                    "d2h_bytes_per_step": B * T * model.odim * 4, "steps": e2e_steps,
                    "ms_per_step": e2e_ms / e2e_steps, "batch_latency": e2e_lat,
                    # what bounds the end-to-end number: the step's input crosses PCIe once (Gen5 x16: ~55 GB/s in practice)
                    "h2d_gb_per_s": ((B * PCM_SAMPLES * 2) if pcm_mode else (B * T * idim * 4)) / (e2e_ms / e2e_steps * 1e-3) / 1e9,
                    "api": ("wekws_b200.Pipeline(Fbank, KWSModel)(pcm) -> wekws_pipeline_forward" if pcm_mode else "wekws_b200.KWSModel.forward(feats, cache)")
                           + "; pinned host input in, posteriors out, H2D double-buffered on a copy stream; "
                             "own step count: warm-up until stable (>= 0.5 s), then >= 1 s timed"},
            "gpu_launches": launches, "tensor_cores": tc,
            "roofline": {"kernel": ("fbank_kernel + " if pcm_mode else "") + kname, "bound": "hbm",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": peak_src + ", burst", "traffic": traffic,
                         "algorithmic_bytes_per_frame": bpf, "launch_ms": launch_ms,
                         "fp32_tflops": (flop_per_frame * B * T / (launch_ms * 1e-3) / 1e12) if flop_per_frame else None,
                         "note": "HBM fraction as SURVEY 8d asks; at fp32 parity the fused backbones are bound by "
                                 "instruction issue / shared memory / the tensor pipe (DESIGN.md section 4)"},
        }
        # SURVEY 8d second figure for the tensor-core kernels: bf16 tensor-pipe utilisation = dense GEMM FLOP/frame
        # x 3 passes of the bf16x3 split / measured bf16 peak (MEASURED_PEAKS.json)
        dense = {"mdtc": 34 * 2 * 64 * 64 + 2 * 80 * 64, "tcn": 32 * 2 * 64 * 64 + 2 * 80 * 64,
                 "ds_tcn": 4 * 2 * 256 * 256 + 2 * 80 * 256}.get(model_name)
        bf16_peak = float(peaks.get("bf16_tflops", 0) or 0)
        if dense and tc and not pcm_mode and bf16_peak:
            tf = 3.0 * dense * B * T / (launch_ms * 1e-3) / 1e12
            res["roofline"]["tensor_pipe"] = {"achieved_bf16_tflops": tf, "peak_bf16_tflops": bf16_peak,
                                              "frac": tf / bf16_peak, "passes": 3}
        return res


def cpu_baseline_subprocess(workload, orig_affinity, budget_s):
    """The CPU leg in a fresh process with the full CPU set (this process is pinned to its GPU's NUMA node)."""
    cur = None
    try:
        if orig_affinity:
            cur = os.sched_getaffinity(0)
            os.sched_setaffinity(0, orig_affinity)
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload,
                              "--steps", "40", "--warmup", "2", "--cpu-budget", str(budget_s)],
                             capture_output=True, text=True, timeout=600,
                             env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        line = [ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)["cpu_baseline"]
    except Exception as e:
        return {"value": None, "unit": "audio-hours/s", "cores": 0, "kind": "port", "sample": f"failed: {e!r}"}
    finally:
        if cur:
            os.sched_setaffinity(0, cur)


class _OnlyTheLine:
    """The driver reads ONE JSON line from stdout.  Libraries write there too (NCCL prints its version line on the boxes
    where NCCL_DEBUG is set), so everything else of this process is sent to stderr: fd 1 is pointed at fd 2 for the
    whole run and the line is written to the saved descriptor at the end."""

    def __init__(self):
        sys.stdout.flush()
        self.fd = os.dup(1)
        os.dup2(2, 1)

    def emit(self, obj):
        sys.stdout.flush()
        os.write(self.fd, (json.dumps(obj) + "\n").encode())


def main():
    out = _OnlyTheLine()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="mdtc_b1024_t40", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra_workloads (BASELINE configs[2..4])")
    ap.add_argument("--cpu-budget", type=float, default=60.0, help="seconds of timed CPU work for --impl reference")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    config = workload_config(args.workload, args.gpus)

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_reference_run(args.workload, args.steps, args.warmup, budget_s=args.cpu_budget)
        out.emit(reference_line(args, config, r))
        return 0

    placement, orig_aff = bind_to_gpu_cpus(local)
    import torch
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (B200)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=dev)
    runner = Runner(dev, rank, world, dist)
    main_res = runner.run(args.workload, args.steps, args.warmup, dump_dir=args.dump_outputs)
    extras = []
    if not args.no_extras and args.workload == "mdtc_b1024_t40":
        for w in EXTRAS:
            r = runner.run(w, steps=0, warmup=5, min_region_s=0.25)
            if r is not None:
                extras.append(r)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    line = {"metric": METRIC, "value": main_res["value"], "unit": "audio-hours/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
            "config": dict(config, host_placement=placement)}
    for k in ("frames_per_sec", "p50_step_latency_ms", "p99_step_latency_ms", "p50_chunk_latency_ms_1stream", "clocks",
              "e2e", "gpu_launches", "tensor_cores", "roofline"):
        line[k] = main_res[k]
    if extras:
        line["extra_workloads"] = extras
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_subprocess(args.workload, orig_aff, budget_s=15.0)
    out.emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
