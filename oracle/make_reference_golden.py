#!/usr/bin/env python
"""Golden vectors recorded from the reference itself (test infrastructure), so that the tests that compare with it run
without a reference checkout:

    python oracle/make_reference_golden.py <reference checkout>

Larger outputs are stored as a fixed, seeded sample (the sample's positions travel with it) to keep the files small.

* tests/golden/stream23.npz: the reference's KWSModel (wekws/model/kws_model.py) for every tests/cases.py case, three
  23-frame chunks of the same input streamed back to back with the cache carried: every output, and the cache at 256
  positions that hold data after the third chunk.
* tests/golden/kaldi_live.npz: torchaudio.compliance.kaldi.fbank / .mfcc (the functions the reference's data
  pipeline calls) on 3 s and 2 s of synthetic audio: 40 frames of each.
* tests/golden/runtime_fbank.npz: the reference's C++ front-end (runtime/core/frontend/fbank.h, fft.cc), built by
  oracle/Makefile into oracle/_ref/ref_fbank, on 2 s of synthetic audio (40 of its frames) and on 399 samples (no
  whole frame).
* tests/golden/checkpoint_schema.npz: key, shape and dtype of every state_dict entry of the reference's model for
  each shipped config.
"""
import contextlib
import io
import os
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden")
STREAM_T, STREAM_STEPS, CACHE_SAMPLES, FRAME_SAMPLES = 23, 3, 256, 40
CKPT_MODELS = ("mdtc", "mdtc_small", "ds_tcn", "tcn", "gru")


def frame_sample(n, seed):
    g = np.random.default_rng(seed)
    return np.sort(g.choice(n, size=min(n, FRAME_SAMPLES), replace=False)).astype(np.int64)


def gen_model_stream():
    from wekws.model.kws_model import init_model
    from tests.cases import CASE_NAMES, build_model
    from wekws_b200 import synth
    arrays = {}
    for ci, case in enumerate(CASE_NAMES):
        cfg, ref, B = build_model(case, init_model)
        gru = cfg["backbone"]["type"] == "gru"
        x = synth.features(B, STREAM_T, cfg["input_dim"], seed=5, cmvn_like=ref.global_cmvn is not None)
        cache = torch.zeros(cfg["backbone"]["num_layers"], B, cfg["hidden_dim"]) if gru else torch.zeros(0, 0, 0)
        arrays[f"{case}_digest"] = np.float64(synth.state_digest(ref))
        arrays[f"{case}_x_sum"] = np.float64(x.double().sum())
        caches = []
        with torch.no_grad():
            for i in range(STREAM_STEPS):
                y, cache = ref(x, cache)
                arrays[f"{case}_y{i}"] = y.numpy()
                caches.append(cache.numpy().reshape(-1))
        live = np.flatnonzero(caches[-1])
        idx = np.sort(np.random.default_rng(ci).permutation(live)[:CACHE_SAMPLES]).astype(np.int64)
        arrays[f"{case}_cshape"] = np.array(cache.shape, dtype=np.int64)
        arrays[f"{case}_cidx"] = idx
        for i, c in enumerate(caches):
            arrays[f"{case}_c{i}"] = c[idx]
    np.savez_compressed(os.path.join(OUT, "stream23.npz"), **arrays)


def gen_kaldi_live():
    import torchaudio.compliance.kaldi as kaldi
    from wekws_b200 import synth
    fb = synth.pcm_int16(1, 16000 * 3, seed=77)[0].float()
    mf = synth.pcm_int16(1, 16000 * 2, seed=78)[0].float()
    fbank = kaldi.fbank(fb.unsqueeze(0), num_mel_bins=80, frame_length=25, frame_shift=10, dither=0.0,
                        energy_floor=0.0, sample_frequency=16000).numpy()
    mfcc = kaldi.mfcc(mf.unsqueeze(0), num_ceps=80, num_mel_bins=80, frame_length=25, frame_shift=10, dither=0.0,
                      energy_floor=0.0, sample_frequency=16000).numpy()
    arrays = {}
    for name, f, seed in (("fbank80_seed77", fbank, 77), ("mfcc80_seed78", mfcc, 78)):
        idx = frame_sample(f.shape[0], seed)
        arrays[name + "_shape"] = np.array(f.shape, dtype=np.int64)
        arrays[name + "_frames"] = idx
        arrays[name] = f[idx]
    np.savez_compressed(os.path.join(OUT, "kaldi_live.npz"), **arrays)


def gen_runtime_fbank(ref_root):
    from wekws_b200 import synth
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "REF=" + os.path.join(ref_root, "runtime", "core")],
                   check=True)
    binary = os.path.join(ROOT, "oracle", "_ref", "ref_fbank")
    wave = synth.pcm_int16(1, 16000 * 2, seed=4)[0].float()
    arrays = {}
    with tempfile.TemporaryDirectory() as tmp:
        fin, fout = os.path.join(tmp, "in.f32"), os.path.join(tmp, "out.f32")

        def run(w, num_bins):
            w.numpy().astype("<f4").tofile(fin)
            subprocess.run([binary, str(num_bins), fin, fout], check=True)
            return np.fromfile(fout, dtype="<f4").reshape(-1, num_bins)
        for num_bins in (80, 40):
            f = run(wave, num_bins)
            idx = frame_sample(f.shape[0], num_bins)
            arrays[f"fbank{num_bins}_shape"] = np.array(f.shape, dtype=np.int64)
            arrays[f"fbank{num_bins}_frames"] = idx
            arrays[f"fbank{num_bins}"] = f[idx]
            arrays[f"fbank{num_bins}_399_shape"] = np.array(run(wave[:399], num_bins).shape, dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "runtime_fbank.npz"), **arrays)


def gen_checkpoint_schema():
    from wekws.model.kws_model import init_model
    from wekws_b200.configs import model_config
    arrays = {}
    for name in CKPT_MODELS:
        with contextlib.redirect_stdout(io.StringIO()):
            sd = init_model(model_config(name)).state_dict()
        keys = sorted(sd)
        arrays[f"{name}_keys"] = np.array(keys)
        arrays[f"{name}_dtypes"] = np.array([str(sd[k].dtype).replace("torch.", "") for k in keys])
        arrays[f"{name}_ndim"] = np.array([sd[k].dim() for k in keys], dtype=np.int64)
        arrays[f"{name}_dims"] = np.array([d for k in keys for d in sd[k].shape], dtype=np.int64)
    np.savez_compressed(os.path.join(OUT, "checkpoint_schema.npz"), **arrays)


def main():
    if len(sys.argv) != 2 or not os.path.isdir(os.path.join(sys.argv[1], "wekws")):
        sys.exit("usage: python oracle/make_reference_golden.py <reference checkout>")
    ref_root = os.path.abspath(sys.argv[1])
    sys.path.insert(0, ROOT)
    sys.path.insert(0, ref_root)
    gen_model_stream()
    gen_kaldi_live()
    gen_runtime_fbank(ref_root)
    gen_checkpoint_schema()
    for name in ("stream23", "kaldi_live", "runtime_fbank", "checkpoint_schema"):
        path = os.path.join(OUT, name + ".npz")
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
