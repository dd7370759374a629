"""Raw PCM -> posteriors in one native call (the composition the reference's callers perform by hand:
``feats = accept_wave(wave); logits, cache = model(feats, cache)``, wekws/bin/stream_kws_ctc.py:482-487, and
score.py's dataset front-end + ``model(feats)``, score.py:117-127).

``Pipeline(frontend, model)(pcm, cache)`` goes through ``wekws_pipeline_forward`` of the C ABI: the front-end kernel
and the fused model kernel are launched back to back on the caller's stream with the feature tensor pinned in L2 by
a persisting access-policy window, so the (B, frames, idim) features are produced and consumed on chip.
"""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import torch

from . import _native
from .frontend import Fbank
from .kws_model import KWSModel, _EMPTY


class Pipeline:
    def __init__(self, frontend: Fbank, model: KWSModel):
        if frontend.feature_dim != model.idim:
            raise ValueError(f"the front-end produces {frontend.feature_dim} features, the model expects {model.idim}")
        self.frontend, self.model = frontend, model
        self._scratch = None

    def __call__(self, pcm: torch.Tensor, in_cache: torch.Tensor = _EMPTY, softmax: bool = False
                 ) -> Tuple[torch.Tensor, torch.Tensor]:
        m, fe = self.model, self.frontend
        if not pcm.is_cuda:
            raise RuntimeError("wekws_b200.Pipeline runs on CUDA (sm_100a) only; got a CPU tensor (no CPU fallback)")
        if m.training:
            raise RuntimeError("wekws_b200.KWSModel is inference-only: call model.eval() first")
        if pcm.dim() != 2 or pcm.dtype not in (torch.int16, torch.float32):
            raise ValueError("pcm must be a (B, N) int16 or float32 tensor in int16 scale")
        if pcm.stride(1) != 1:
            pcm = pcm.contiguous()
        dev = pcm.device
        B, N = pcm.shape
        T = fe.num_frames(N)
        h_model, in_cache, out, out_cache = m._prepare_call(dev, B, T, in_cache)
        cache_ptr = None if in_cache is None else in_cache.data_ptr()
        if T == 0 or B == 0:
            return out, out_cache
        need = B * T * m.idim
        if self._scratch is None or self._scratch.numel() < need or self._scratch.device != dev:
            self._scratch = torch.empty(need, device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            rc = _native.lib().wekws_pipeline_forward(
                fe._handle(dev), h_model, C.c_void_p(pcm.data_ptr()),
                _native.PCM_S16 if pcm.dtype == torch.int16 else _native.PCM_F32, B, N, pcm.stride(0),
                C.c_void_p(self._scratch.data_ptr()), cache_ptr, C.c_void_p(out.data_ptr()),
                C.c_void_p(out_cache.data_ptr()), _native.FWD_SOFTMAX if softmax else 0,
                C.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
        _native.check(rc, "wekws_pipeline_forward")
        return out, out_cache
