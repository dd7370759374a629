"""wekws_b200 -- B200-native (sm_100a) streaming keyword-spotting forward path for WeKws.

Public surface mirrors the reference (wenet-e2e/wekws):
    init_model, KWSModel     <- wekws/model/kws_model.py
    Fbank, fbank             <- torchaudio.compliance.kaldi.fbank as the reference calls it
    Mfcc, mfcc               <- torchaudio.compliance.kaldi.mfcc  (processor.py:157-166, the mdtc configs' front-end)
    load_cmvn, load_kaldi_cmvn <- wekws/utils/cmvn.py
    Pipeline(frontend, model) <- raw PCM -> posteriors in one native call (stream_kws_ctc.py:482-487 composition)
    patch_reference()        -> makes `wekws.model.kws_model` resolve to this implementation
    det_stats, det_curve     <- wekws/bin/compute_det.py threshold sweep (on the device, bit-exact)
    ctc_prefix_beam_search, ctc_keyword_hits, write_ctc_scores <- wekws/model/loss.py:206-312 + score_ctc.py:198-226
    context_expansion        <- wekws/dataset/processor.py context_expansion + frame_skip (FSMN / CTC recipes)
    KeyWordSpotter           <- wekws/bin/stream_kws_ctc.py KeyWordSpotter: PCM chunks -> detections, B streams at once
    export_native()          -> weight file for the C++ runtime shim (the role of wekws/bin/export_onnx.py)
    export_onnx()            <- wekws/bin/export_onnx.py: the ONNX file (input, cache -> output, r_cache) for the ORT runtime
"""
from .cmvn import load_cmvn, load_kaldi_cmvn
from .configs import MODEL_NAMES, model_config
from .frontend import Fbank, Mfcc, fbank, mfcc
from .kws_model import GlobalCMVN, KWSModel, init_model
from .ctc import ctc_keyword_hits, ctc_prefix_beam_search, ctc_state, write_ctc_scores
from .export import export_native
from .export_onnx import export_onnx
from .overlay import patch_reference
from .pipeline import Pipeline
from .postproc import context_expansion, det_curve, det_stats, det_thresholds
from .spotter import KeyWordSpotter

__all__ = ["init_model", "KWSModel", "GlobalCMVN", "Fbank", "fbank", "Mfcc", "mfcc", "load_cmvn", "load_kaldi_cmvn",
           "model_config", "MODEL_NAMES", "patch_reference", "export_native", "export_onnx", "det_stats", "det_curve", "det_thresholds", "context_expansion",
           "Pipeline", "ctc_prefix_beam_search", "ctc_keyword_hits", "ctc_state", "write_ctc_scores", "KeyWordSpotter"]
__version__ = "0.1.0"
