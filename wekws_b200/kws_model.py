"""Drop-in ``KWSModel`` / ``init_model`` for the reference's wekws/model/kws_model.py.

Same constructor, attributes (``idim``, ``odim``, ``hdim``, ``backbone.padding``), the same
``state_dict`` key set and shapes (so reference checkpoints load with ``strict=True`` and
``wekws/bin/average_model.py`` output loads too), and the same call surface:

    logits, out_cache = model(feats)               # wekws/bin/score.py:125
    logits, cache     = model(feats, cache)        # wekws/bin/stream_kws_ctc.py:487

The modules in here are parameter HOLDERS only.  ``forward`` hands raw device pointers to
the C-ABI library (include/wekws_b200.h) whose fused sm_100a kernels do all the work:
CMVN -> Linear+ReLU -> backbone with streaming cache -> classifier -> activation
(kws_model.py:65-76).  There is no PyTorch / CPU fallback: CPU tensors, training mode or a
missing native library raise.
"""
from __future__ import annotations

import ctypes as C
import sys
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import _native
from .cmvn import load_cmvn, load_kaldi_cmvn

_EMPTY = torch.zeros(0, 0, 0, dtype=torch.float)


def _holder(**children) -> nn.Module:
    m = nn.Module()
    for name, child in children.items():
        m.add_module(name, child)
    return m


class GlobalCMVN(nn.Module):
    """Buffers of wekws/model/cmvn.py:19-35; applied inside the fused kernel."""

    def __init__(self, mean: torch.Tensor, istd: torch.Tensor, norm_var: bool = True):
        super().__init__()
        assert mean.shape == istd.shape
        self.norm_var = norm_var
        self.register_buffer("mean", mean)
        self.register_buffer("istd", istd)


def _linear_subsampling(idim: int, odim: int) -> nn.Module:
    """state_dict: out.0.{weight,bias} (subsampling.py:45-48)."""
    m = _holder(out=nn.Sequential(nn.Linear(idim, odim), nn.ReLU()))
    m.subsampling_rate = 1
    return m


def _mdtc_block(ch: int, k: int, d: int) -> nn.Module:
    """conv1.{conv,bn,pointwise}, bn1, conv2, bn2 (mdtc.py:37-53, 79-92)."""
    blk = _holder(
        conv1=_holder(conv=nn.Conv1d(ch, ch, k, dilation=d, groups=ch), bn=nn.BatchNorm1d(ch),
                      pointwise=nn.Conv1d(ch, ch, 1)),
        bn1=nn.BatchNorm1d(ch), conv2=nn.Conv1d(ch, ch, 1), bn2=nn.BatchNorm1d(ch))
    blk.padding = d * (k - 1)
    return blk


def _mdtc(num_stack: int, stack_size: int, ch: int, k: int) -> nn.Module:
    """preprocessor + blocks.{s}.res_blocks.{l} with dilations 2**l (mdtc.py:151-156, 226-238)."""
    assert k % 2 == 1
    pre = _mdtc_block(ch, k, 1)
    stacks = nn.ModuleList()
    padding = pre.padding
    for _ in range(num_stack):
        res = nn.ModuleList([_mdtc_block(ch, k, 2 ** l) for l in range(stack_size)])
        st = _holder(res_blocks=res)
        st.padding = sum(b.padding for b in res)
        padding += st.padding
        stacks.append(st)
    bb = _holder(preprocessor=pre, blocks=stacks)
    bb.padding = padding
    bb.half_padding = padding // 2
    bb.kind, bb.num_stack, bb.stack_size, bb.kernel_size = "mdtc", num_stack, stack_size, k
    return bb


def _tcn(num_layers: int, ch: int, k: int, dropout: float, ds: bool) -> nn.Module:
    """network.{i}.cnn.{0,1[,3,4]} with dilation 2**i (tcn.py:75-84, 101-114, 133-137)."""
    net = nn.ModuleList()
    padding = 0
    for i in range(num_layers):
        d = 2 ** i
        if ds:
            cnn = nn.Sequential(nn.Conv1d(ch, ch, k, dilation=d, groups=ch), nn.BatchNorm1d(ch), nn.ReLU(),
                                nn.Conv1d(ch, ch, 1), nn.BatchNorm1d(ch), nn.ReLU(), nn.Dropout(dropout))
        else:
            cnn = nn.Sequential(nn.Conv1d(ch, ch, k, dilation=d), nn.BatchNorm1d(ch), nn.ReLU(),
                                nn.Dropout(dropout))
        blk = _holder(cnn=cnn)
        blk.padding = (k - 1) * d
        padding += blk.padding
        net.append(blk)
    bb = _holder(network=net)
    bb.padding = padding
    bb.kind, bb.num_layers, bb.kernel_size, bb.ds = ("ds_tcn" if ds else "tcn"), num_layers, k, ds
    return bb


def _affine(idim: int, odim: int, bias: bool = True) -> nn.Module:
    """AffineTransform / LinearTransform: state_dict linear.{weight[,bias]} (fsmn.py:56-60, 114-118)."""
    return _holder(linear=nn.Linear(idim, odim, bias=bias))


def _fsmn(input_dim: int, input_affine_dim: int, fsmn_layers: int, linear_dim: int, proj_dim: int, lorder: int,
          rorder: int, lstride: int, rstride: int, output_affine_dim: int, output_dim: int) -> nn.Module:
    """Parameter holder with the key set of wekws/model/fsmn.py FSMN (fsmn.py:401-456): in_linear{1,2}.linear.*,
    fsmn.{l}.0.linear.weight (LinearTransform, no bias), fsmn.{l}.1.conv_{left,right}.weight (FSMNBlock: depthwise
    Conv2d (proj,1,order,1), no bias), fsmn.{l}.2.linear.* (AffineTransform), out_linear{1,2}.linear.*.  The blocks
    are built with strides (1, 1) whatever the config says, exactly as _build_repeats does (fsmn.py:384-391);
    lstride / rstride only enter `padding`."""
    if rorder < 1:
        raise NotImplementedError("wekws_b200: FSMN right_order must be >= 1 (the reference's FSMNBlock.forward itself "
                                  "fails for right_order = 0, fsmn.py:235)")
    layers = []
    for _ in range(fsmn_layers):
        mem = _holder(conv_left=nn.Conv2d(proj_dim, proj_dim, [lorder, 1], dilation=[1, 1], groups=proj_dim, bias=False),
                      conv_right=nn.Conv2d(proj_dim, proj_dim, [rorder, 1], dilation=[1, 1], groups=proj_dim, bias=False))
        layers.append(nn.Sequential(_affine(linear_dim, proj_dim, bias=False), mem, _affine(proj_dim, linear_dim),
                                    nn.Module()))
    bb = _holder(in_linear1=_affine(input_dim, input_affine_dim), in_linear2=_affine(input_affine_dim, linear_dim),
                 relu=nn.Module(), fsmn=nn.Sequential(*layers), out_linear1=_affine(linear_dim, output_affine_dim),
                 out_linear2=_affine(output_affine_dim, output_dim))
    bb.kind = "fsmn"
    bb.input_dim, bb.input_affine_dim, bb.fsmn_layers, bb.linear_dim, bb.proj_dim = \
        input_dim, input_affine_dim, fsmn_layers, linear_dim, proj_dim
    bb.lorder, bb.rorder, bb.lstride, bb.rstride = lorder, rorder, lstride, rstride
    bb.output_affine_dim, bb.output_dim = output_affine_dim, output_dim
    bb.padding = (lorder - 1) * lstride + rorder * rstride          # fsmn.py:443-444 (API attribute)
    bb.cache_len = (lorder - 1) + rorder                            # what the blocks really keep (strides 1, 1)
    return bb


def _linear_classifier(idim: int, odim: int) -> nn.Module:
    """state_dict: linear.{weight,bias} (classifier.py:57-61)."""
    return _holder(linear=nn.Linear(idim, odim))


class KWSModel(nn.Module):
    """wekws/model/kws_model.py:33-95, executed by libwekws_b200.so."""

    def __init__(self, idim: int, odim: int, hdim: int, global_cmvn: Optional[nn.Module],
                 preprocessing: Optional[nn.Module], backbone: nn.Module, classifier: nn.Module,
                 activation: nn.Module):
        super().__init__()
        self.idim, self.odim, self.hdim = idim, odim, hdim
        self.global_cmvn = global_cmvn
        self.preprocessing = preprocessing
        self.backbone = backbone
        self.classifier = classifier
        self.activation = activation
        self._handle = None          # wekws_model*
        self._handle_dev = None
        self._dirty = True
        # "auto": tcgen05 tensor cores (3-pass bf16 split, ~1e-5 of fp32) where a fused kernel exists,
        # FP32 FMA elsewhere; "fp32": FP32 FMA kernels only.
        self.precision = "auto"
        self._precision_applied = None

    # ---------------------------------------------------------------- weight life-cycle
    def invalidate(self) -> None:
        """Forces a re-pack.  Normally not needed: in-place edits are detected through the tensors' version counters
        (``_fingerprint``); only writes that bypass autograd's counter (``.data_ptr()`` pokes) need this."""
        self._dirty = True

    def load_state_dict(self, *args, **kwargs):
        self._dirty = True
        return super().load_state_dict(*args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self._dirty = True
        return super()._apply(fn, *args, **kwargs)

    def _release(self) -> None:
        h = self.__dict__.get("_handle")
        if h is not None:
            try:
                _native.lib().wekws_model_destroy(h)
            except Exception:
                pass
            self.__dict__["_handle"] = None

    def __del__(self):
        self._release()

    def __getstate__(self):      # the native handle is rebuilt lazily after copy / unpickle
        state = self.__dict__.copy()
        state["_handle"], state["_handle_dev"], state["_dirty"] = None, None, True
        state["_precision_applied"] = None
        state.pop("_packed_fp", None)
        state.pop("_packed_tensors", None)
        return state

    def _native_config(self) -> _native.ModelConfig:
        bb = self.backbone
        cfg = _native.ModelConfig()
        cfg.idim, cfg.hdim, cfg.odim = self.idim, self.hdim, self.odim
        if isinstance(bb, nn.GRU):
            if not (bb.batch_first and not bb.bidirectional and bb.bias and bb.input_size == bb.hidden_size):
                raise NotImplementedError("wekws_b200: only GRU(hdim, hdim, batch_first=True) is supported")
            cfg.backbone, cfg.num_layers, cfg.hdim = _native.BACKBONE_GRU, bb.num_layers, bb.hidden_size
        elif getattr(bb, "kind", None) == "mdtc":
            cfg.backbone = _native.BACKBONE_MDTC
            cfg.num_stack, cfg.stack_size, cfg.kernel_size = bb.num_stack, bb.stack_size, bb.kernel_size
        elif getattr(bb, "kind", None) in ("tcn", "ds_tcn"):
            cfg.backbone = _native.BACKBONE_DSTCN if bb.ds else _native.BACKBONE_TCN
            cfg.num_layers, cfg.kernel_size = bb.num_layers, bb.kernel_size
        elif getattr(bb, "kind", None) == "fsmn":
            if self.preprocessing is not None and not getattr(self.preprocessing, "is_identity", False):
                raise NotImplementedError("wekws_b200: FSMN runs with preprocessing type 'none' (as every shipped config)")
            if not isinstance(self.classifier, nn.Identity):
                raise NotImplementedError("wekws_b200: FSMN runs with classifier type 'identity' (as every shipped config)")
            cfg.backbone, cfg.num_layers = _native.BACKBONE_FSMN, bb.fsmn_layers
            cfg.fsmn_input_affine_dim, cfg.fsmn_linear_dim, cfg.fsmn_proj_dim = bb.input_affine_dim, bb.linear_dim, bb.proj_dim
            cfg.fsmn_left_order, cfg.fsmn_right_order, cfg.fsmn_output_affine_dim = bb.lorder, bb.rorder, bb.output_affine_dim
        else:
            raise NotImplementedError(f"wekws_b200: backbone {type(bb).__name__} has no fused kernel")
        if isinstance(self.activation, nn.Sigmoid):
            cfg.activation = _native.ACT_SIGMOID
        elif isinstance(self.activation, nn.Identity):
            cfg.activation = _native.ACT_IDENTITY
        else:
            raise NotImplementedError("wekws_b200: activation must be nn.Sigmoid or nn.Identity")
        cfg.norm_var = 1 if (self.global_cmvn is None or self.global_cmvn.norm_var) else 0
        return cfg

    def _build_handle(self, finalize: bool = True):
        """Creates the native model and feeds it the state_dict by its reference key names."""
        lib = _native.lib()
        self._release()
        cfg = self._native_config()
        h = C.c_void_p()
        _native.check(lib.wekws_model_create(C.byref(cfg), C.byref(h)), "wekws_model_create")
        self._handle = h
        for name, t in self.state_dict().items():
            if name.endswith("num_batches_tracked"):
                continue
            host = t.detach().to(device="cpu", dtype=torch.float32).contiguous()
            _native.check(lib.wekws_model_set_tensor(h, name.encode(), C.c_void_p(host.data_ptr()), host.numel()),
                          f"wekws_model_set_tensor({name})")
        if finalize:
            _native.check(lib.wekws_model_finalize(h), "wekws_model_finalize")
        else:
            _native.check(lib.wekws_model_pack(h), "wekws_model_pack")
        return h

    def _fingerprint(self) -> int:
        """Sum of the in-place version counters of the tensors the pack was made from: changes on optimizer steps,
        `.copy_`, `backbone.load_state_dict(...)`, weight surgery.  The tensor list is cached at pack time (15 us for
        the 361 tensors of mdtc, < 1 us for GRU); replacing a Parameter OBJECT needs invalidate()."""
        lst = self.__dict__.get("_packed_tensors")
        return -1 if lst is None else sum([t._version for t in lst])

    def _ensure(self, device: torch.device):
        if (self._dirty or self._handle is None or self._handle_dev != device
                or self._fingerprint() != self.__dict__.get("_packed_fp")):
            with torch.cuda.device(device):
                self._build_handle(finalize=True)
            self._handle_dev = device
            self._dirty = False
            self._precision_applied = None
            self.__dict__["_packed_tensors"] = list(self.parameters()) + list(self.buffers())
            self.__dict__["_packed_fp"] = self._fingerprint()
        return self._handle

    def uses_tensor_cores(self, T: int, B: int = None) -> bool:
        '''True if a forward with T frames per call (and, for the GRU, B streams) takes the tcgen05 kernel (model
        already on a GPU).  Without B the answer is for a large batch.'''
        if self._handle is None or self._dirty or self.precision == "fp32":
            return False
        self._apply_precision(self._handle)
        if B is None:
            return bool(_native.lib().wekws_model_uses_tensor_cores(self._handle, T))
        return bool(_native.lib().wekws_model_uses_tensor_cores_bt(self._handle, B, T))

    _PRECISIONS = {"auto": 0, "fp32": 1, "tensor": 2}

    def _apply_precision(self, h):
        if self._precision_applied != self.precision:
            if self.precision not in self._PRECISIONS:
                raise ValueError("precision must be 'auto', 'fp32' or 'tensor'")
            _native.check(_native.lib().wekws_model_set_precision(h, self._PRECISIONS[self.precision]),
                          "wekws_model_set_precision")
            self._precision_applied = self.precision


    # ------------------------------------------------------------------------- forward
    def _prepare_call(self, dev: torch.device, B: int, T: int, in_cache: torch.Tensor):
        """What every native forward (``model(feats)`` and ``Pipeline``) needs for B streams of T frames on `dev`: the
        handle, packed and with the precision applied; the input cache as a contiguous fp32 tensor on `dev` (None: start
        of stream; the caller keeps it alive until the launch); the output tensors.  For T == 0 the output cache is the
        input cache (or zeros)."""
        if isinstance(self.backbone, nn.GRU):
            cache_shape = (self.backbone.num_layers, B, self.hdim)
        elif getattr(self.backbone, "kind", None) == "fsmn":      # 4-D: one column block per layer (fsmn.py:488)
            cache_shape = (B, self.backbone.proj_dim, self.backbone.cache_len, self.backbone.fsmn_layers)
        else:
            cache_shape = (B, self.hdim, self.backbone.padding)
        if in_cache is not None and in_cache.numel() > 0:
            if tuple(in_cache.shape) != cache_shape:
                raise ValueError(f"in_cache must be {cache_shape}, got {tuple(in_cache.shape)}")
            if in_cache.device != dev or in_cache.dtype != torch.float32 or not in_cache.is_contiguous():
                in_cache = in_cache.to(device=dev, dtype=torch.float32).contiguous()
        else:
            in_cache = None
        h = self._ensure(dev)
        self._apply_precision(h)
        out = torch.empty((B, T, self.odim), device=dev, dtype=torch.float32)
        if T == 0 and in_cache is not None:
            out_cache = in_cache.clone()
        elif T == 0:
            out_cache = torch.zeros(cache_shape, device=dev, dtype=torch.float32)
        else:
            out_cache = torch.empty(cache_shape, device=dev, dtype=torch.float32)
        return h, in_cache, out, out_cache

    def _run(self, x: torch.Tensor, in_cache: torch.Tensor, flags: int) -> Tuple[torch.Tensor, torch.Tensor]:
        if self.training:
            raise RuntimeError("wekws_b200.KWSModel is inference-only: call model.eval() first "
                               "(training-mode BatchNorm/Dropout are not implemented)")
        if not x.is_cuda:
            raise RuntimeError("wekws_b200.KWSModel runs on CUDA (sm_100a) only; got a CPU tensor. "
                               "There is no CPU fallback -- move the model and inputs to a B200.")
        if x.dtype != torch.float32:
            raise TypeError(f"wekws_b200.KWSModel expects float32 features, got {x.dtype}")
        if x.dim() != 3 or x.size(2) != self.idim:
            raise ValueError(f"features must be (B, T, {self.idim}), got {tuple(x.shape)}")
        dev = x.device
        B, T = x.size(0), x.size(1)
        if not x.is_contiguous():
            x = x.contiguous()
        h, in_cache, out, out_cache = self._prepare_call(dev, B, T, in_cache)
        cache_ptr = None if in_cache is None else in_cache.data_ptr()
        if B > 0 and T > 0:
            fwd = _native.lib().wekws_model_forward
            if torch.cuda.current_device() == dev.index:          # common case: no device switch needed
                rc = fwd(h, x.data_ptr(), cache_ptr, out.data_ptr(), out_cache.data_ptr(), B, T, flags,
                         torch.cuda.current_stream(dev).cuda_stream)
            else:
                with torch.cuda.device(dev):
                    rc = fwd(h, x.data_ptr(), cache_ptr, out.data_ptr(), out_cache.data_ptr(), B, T, flags,
                             torch.cuda.current_stream(dev).cuda_stream)
            if rc != 0:
                _native.check(rc, "wekws_model_forward")
        return out, out_cache

    def forward(self, x: torch.Tensor, in_cache: torch.Tensor = _EMPTY) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run(x, in_cache, 0)

    def forward_softmax(self, x: torch.Tensor, in_cache: torch.Tensor = _EMPTY) -> Tuple[torch.Tensor, torch.Tensor]:
        """kws_model.py:78-90 -- softmax over the output dim after the activation."""
        return self._run(x, in_cache, _native.FWD_SOFTMAX)

    def fuse_modules(self):
        """The reference fuses conv+bn+relu for int8 PTQ (static_quantize.py:94); here every
        BatchNorm is already folded natively at pack time, so there is nothing to do."""
        return None


def init_model(configs: dict) -> KWSModel:
    """Config -> model factory with the reference's keys and defaults (kws_model.py:97-214)."""
    cmvn = configs.get("cmvn", {})
    if "cmvn_file" in cmvn and cmvn["cmvn_file"] is not None:
        loader = load_kaldi_cmvn if "kaldi" in cmvn["cmvn_file"] else load_cmvn
        mean, istd = loader(cmvn["cmvn_file"])
        global_cmvn = GlobalCMVN(torch.from_numpy(mean).float(), torch.from_numpy(istd).float(), cmvn["norm_var"])
    else:
        global_cmvn = None

    input_dim, output_dim, hidden_dim = configs["input_dim"], configs["output_dim"], configs["hidden_dim"]

    prep_type = configs["preprocessing"]["type"]
    if prep_type == "linear":
        preprocessing = _linear_subsampling(input_dim, hidden_dim)
    elif prep_type == "none" and configs["backbone"]["type"] == "fsmn":
        preprocessing = nn.Module()          # NoSubsampling (subsampling.py:28-39): identity, no parameters
        preprocessing.subsampling_rate, preprocessing.is_identity = 1, True
    elif prep_type in ("cnn1d_s1", "none"):
        raise NotImplementedError(f"wekws_b200: preprocessing type '{prep_type}' is outside the fused hot path "
                                  "(SURVEY.md section 2 row 4); 'linear' (and 'none' in front of FSMN) are implemented")
    else:
        print("Unknown preprocessing type {}".format(prep_type))
        sys.exit(1)

    bb = configs["backbone"]
    if bb["type"] == "gru":
        backbone = nn.GRU(hidden_dim, hidden_dim, num_layers=bb["num_layers"], batch_first=True)
    elif bb["type"] == "tcn":
        backbone = _tcn(bb["num_layers"], hidden_dim, bb.get("kernel_size", 8), bb.get("dropout", 0.1),
                        bb.get("ds", False))
    elif bb["type"] == "mdtc":
        hidden_dim = bb["hidden_dim"]
        assert bb["causal"] is True, "we now only support causal mdtc"
        backbone = _mdtc(bb["num_stack"], bb["stack_size"], hidden_dim, bb["kernel_size"])
    elif bb["type"] == "fsmn":                                  # kws_model.py:158-170
        backbone = _fsmn(input_dim, bb["input_affine_dim"], bb["num_layers"], bb["linear_dim"], bb["proj_dim"],
                         bb["left_order"], bb["right_order"], bb["left_stride"], bb["right_stride"],
                         bb["output_affine_dim"], output_dim)
    else:
        print("Unknown body type {}".format(bb["type"]))
        sys.exit(1)

    activation: nn.Module = nn.Sigmoid()
    if "classifier" in configs:                                 # kws_model.py:175-195
        classifier_type = configs["classifier"]["type"]
        if classifier_type in ("global", "last"):
            raise NotImplementedError("wekws_b200: the speech-command 'classifier' heads (global/last) are "
                                      "outside the streaming hot path (SURVEY.md section 2 row 8)")
        elif classifier_type == "identity":
            if bb["type"] != "fsmn":
                raise NotImplementedError("wekws_b200: classifier 'identity' is implemented behind the FSMN backbone "
                                          "(the only shipped use, fsmn_ctc.yaml)")
            classifier: nn.Module = nn.Identity()
        else:
            print("Unknown classifier type {}".format(classifier_type))
            sys.exit(1)
        activation = nn.Identity()
    else:
        if bb["type"] == "fsmn":
            raise NotImplementedError("wekws_b200: FSMN needs classifier type 'identity' (its out_linear2 already maps "
                                      "to output_dim, fsmn_ctc.yaml:53-55)")
        classifier = _linear_classifier(hidden_dim, output_dim)
    if "activation" in configs:
        if configs["activation"]["type"] == "identity":
            activation = nn.Identity()
        else:
            print("Unknown activation type {}".format(configs["activation"]["type"]))
            sys.exit(1)
    return KWSModel(input_dim, output_dim, hidden_dim, global_cmvn, preprocessing, backbone, classifier,
                    activation)
