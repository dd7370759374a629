"""Kernel dispatch and call preparation shared by KWSModel and Pipeline: the tensor-core classifier image of the CTC
head (CPU), and the precision a Pipeline call leaves on the model's handle (GPU)."""
import ctypes as C

import numpy as np
import pytest
import torch

from wekws_b200 import Fbank, Pipeline, init_model, model_config, synth


def test_ds_tcn_classifier_image_encodes_the_classifier(native):
    """The ds_tcn CTC head (output_dim 2599) runs as its own tcgen05 GEMM (linear_tc.cu) whose weight image -- 32 KB
    K-major SWIZZLE_128B bf16 hi|lo pieces of 128 output columns x 64 K, [n tile][K slab] -- decodes back to
    classifier.linear.weight: hi = bf16_rn(w), |hi + lo - w| <= 2^-16 |w|, zero beyond N."""
    cfg = model_config("ds_tcn", output_dim=2599)
    model = synth.randomize_(init_model(cfg)).eval()
    h = model._build_handle(finalize=False)
    lib = native.lib()
    N, K = 2599, model.hdim
    ntn, nslab = (N + 127) // 128, K // 64
    n = lib.wekws_model_packed_floats(h, 3)
    assert n * 4 == ntn * nslab * 32768
    raw = torch.empty(n, dtype=torch.float32)
    native.check(lib.wekws_model_packed_copy(h, 3, C.c_void_p(raw.data_ptr()), n), "packed_copy")
    img = raw.numpy().view(np.uint16)
    W = model.state_dict()["classifier.linear.weight"].numpy()
    assert W.shape == (N, K)
    nn, kk = np.meshgrid(np.arange(128), np.arange(64), indexing="ij")
    u16 = (nn * 128 + (((kk >> 3) ^ (nn & 7)) << 4) + (kk & 7) * 2) // 2

    def f(u):
        return (u.astype(np.uint32) << 16).view(np.float32)

    for nt in range(ntn):
        for s in range(nslab):
            base = (nt * nslab + s) * 16384                 # 32 KB piece, in uint16
            hi, lo = f(img[base + u16]), f(img[base + 8192 + u16])
            w = np.zeros((128, 64), np.float32)
            rows = min(128, N - 128 * nt)
            w[:rows] = W[128 * nt:128 * nt + rows, 64 * s:64 * s + 64]
            assert np.array_equal(hi, torch.from_numpy(w).to(torch.bfloat16).float().numpy())
            assert np.all(np.abs(hi + lo - w) <= 2.0 ** -16 * np.abs(w) + 1e-30)
            assert not hi[rows:].any() and not lo[rows:].any()


@pytest.mark.gpu
def test_pipeline_keeps_the_tensor_precision_of_the_model():
    """precision = "tensor" selects the tcgen05 GRU through Pipeline as through model(feats), and a Pipeline call leaves
    the handle in that mode: the next model(feats) is the tensor-core result, bit for bit."""
    dev = "cuda:0"
    cfg = model_config("gru")
    model = synth.randomize_(init_model(cfg), seed=11).eval()
    fresh = init_model(cfg).eval()
    fresh.load_state_dict(model.state_dict())
    model, fresh = model.to(dev), fresh.to(dev)
    model.precision = fresh.precision = "tensor"
    Pipeline(Fbank(cfg["input_dim"]), model)(synth.pcm_int16(16, 6720, seed=1).to(dev))
    assert model.uses_tensor_cores(1, 16)
    x = synth.features(16, 1, cfg["input_dim"], seed=3).to(dev)
    y, c = model(x)
    y_ref, c_ref = fresh(x)
    assert fresh.uses_tensor_cores(1, 16)
    assert torch.equal(y, y_ref) and torch.equal(c, c_ref)
