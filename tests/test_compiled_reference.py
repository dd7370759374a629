"""Checks against the reference's OWN C++ front-end (runtime/core/frontend/fbank.h, fft.cc): what it computed for
the inputs below, compiled by oracle/Makefile and recorded by oracle/make_reference_golden.py in
tests/golden/runtime_fbank.npz (a fixed sample of 40 frames).  It is the Hamming-window variant of the same Fbank
(fbank.h:90-96,164), i.e. what the native runtime feeds the model (feature_pipeline.cc:30-47)."""
import numpy as np
import pytest

from oracle import kws_oracle as O
from tests.conftest import golden
from wekws_b200 import synth


def reference_frontend(num_bins: int):
    """-> (shape of the full output, sampled frame indices, those frames, shape of the output for 399 samples)."""
    g = golden("runtime_fbank")
    key = f"fbank{num_bins}"
    return tuple(g[key + "_shape"]), g[key + "_frames"], g[key], tuple(g[key + "_399_shape"])


@pytest.mark.parametrize("num_bins", [80, 40])
def test_oracle_hamming_matches_compiled_reference(num_bins):
    wave = synth.pcm_int16(1, 16000 * 2, seed=4)[0].float()
    shape, frames, ref, shape_399 = reference_frontend(num_bins)
    out = O.fbank(wave, num_mel_bins=num_bins, window_type="hamming").numpy()
    assert out.shape == shape == (198, num_bins)
    d = np.abs(out[frames] - ref)
    assert d.max() <= 1e-3 and d.mean() <= 2e-5        # two independent fp32 FFTs (SURVEY: 1e-4 typical)
    assert shape_399[0] == 0
    assert O.fbank(wave[:399], num_mel_bins=num_bins, window_type="hamming").shape == shape_399


@pytest.mark.gpu
def test_gpu_hamming_fbank_matches_compiled_reference():
    from wekws_b200 import Fbank
    wave = synth.pcm_int16(1, 16000 * 2, seed=4)[0]
    shape, frames, ref, _ = reference_frontend(80)
    out = Fbank(80, window_type="hamming")(wave.cuda()).cpu().numpy()
    d = np.abs(out[frames] - ref)
    assert out.shape == shape and d.max() <= 1e-3 and d.mean() <= 2e-5
