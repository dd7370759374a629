"""CPU-only tests of the host side: the C-ABI library loads and exports every declared symbol,
BN folding + weight packing (evaluated independently of the kernels), the drop-in Python
surface (state_dict schema, init parity, error behaviour), and the front-end constants."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import kws_oracle as O
from tests import packed_eval as PE
from tests.cases import CASE_NAMES, build_model
from tests.conftest import ROOT, golden
from wekws_b200 import Fbank, init_model, model_config, synth
from wekws_b200 import frontend


def test_library_exports_every_declared_symbol(native):
    hdr = open(os.path.join(ROOT, "include", "wekws_b200.h")).read()
    declared = re.findall(r"^WEKWS_API [\w\s\*]+?\b(wekws_\w+)\(", hdr, flags=re.M)
    assert len(declared) >= 18
    assert sorted(declared) == sorted(native.SIGNATURES), "binding and header disagree"
    lib = C.CDLL(native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} not exported"
    assert native.lib().wekws_abi_version() == native.ABI_VERSION


def test_mfcc_constants_are_bit_identical_to_torchaudio():
    """The DCT matrix and lifter the product uploads are built with torchaudio's own fp32 ops (goldens from
    kaldi._get_dct_matrix / _get_lifter_coeffs, oracle/make_golden.py)."""
    import numpy as np
    from wekws_b200 import frontend
    g = np.load(os.path.join(ROOT, "tests", "golden", "mfcc.npz"))
    assert np.array_equal(frontend.dct_matrix(80, 80).numpy(), g["dct80"])
    assert np.array_equal(frontend.dct_matrix(13, 23).numpy(), g["dct13_23"])
    assert np.array_equal(frontend.lifter_coeffs(80, 22.0).numpy(), g["lifter80"])


def test_native_export_roundtrip_and_runtime_shim_symbols(tmp_path):
    """.wkb exporter (the export_onnx.py role) and the C++ shim's link surface: wekws::KeywordSpotting with the
    reference's public members (runtime/core/kws/keyword_spotting.h:26-55)."""
    import subprocess
    import torch
    from wekws_b200 import export_native, init_model, model_config, synth
    from wekws_b200.export import read_native
    m = synth.randomize_(init_model(model_config("mdtc"))).eval()
    meta = export_native(m, str(tmp_path / "m.wkb"))
    assert meta["cache_dim"] == 64 and meta["cache_len"] == 244
    fields, tensors = read_native(str(tmp_path / "m.wkb"))
    assert fields[:4] == (0, 80, 64, 1)
    sd = {k: v for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    assert set(tensors) == set(sd)
    assert all(torch.equal(tensors[k].reshape(-1), sd[k].float().reshape(-1)) for k in sd)
    so = os.path.join(ROOT, "wekws_b200", "runtime", "libwekws_b200_runtime.so")
    assert os.path.exists(so), "run __graft_entry__.build() first"
    syms = subprocess.run(["nm", "-DC", so], capture_output=True, text=True).stdout
    for want in ("wekws::KeywordSpotting::KeywordSpotting(std::", "wekws::KeywordSpotting::Reset()",
                 "wekws::KeywordSpotting::Forward(std::vector<std::vector<float",
                 "wenet::FeaturePipeline::FeaturePipeline(wenet::FeaturePipelineConfig const&)",
                 "wenet::FeaturePipeline::AcceptWaveform(std::vector<short", "wenet::FeaturePipeline::AcceptWaveform(std::vector<float",
                 "wenet::FeaturePipeline::Read(int, std::vector<std::vector<float", "wenet::FeaturePipeline::set_input_finished()",
                 "wenet::FeaturePipeline::ReadOne(std::vector<float", "wenet::FeaturePipeline::Reset()"):
        assert want in syms, want
    assert os.access(os.path.join(ROOT, "wekws_b200", "runtime", "kws_main_b200"), os.X_OK)


def test_error_reporting_without_gpu(native):
    lib = native.lib()
    h = C.c_void_p()
    bad = native.ModelConfig(backbone=9, idim=80, hdim=64, odim=1)
    assert lib.wekws_model_create(C.byref(bad), C.byref(h)) == -1
    assert "backbone" in native.last_error()
    ok = native.ModelConfig(backbone=native.BACKBONE_MDTC, idim=80, hdim=64, odim=1, num_stack=4, stack_size=4,
                            kernel_size=5, activation=1, norm_var=1)
    assert lib.wekws_model_create(C.byref(ok), C.byref(h)) == 0
    assert lib.wekws_model_padding(h) == 244
    # forward before finalize -> state error, pack with nothing set -> names the missing tensor
    assert lib.wekws_model_forward(h, None, None, None, None, 1, 1, 0, None) == -3
    assert lib.wekws_model_pack(h) == -3
    assert "preprocessing.out.0.weight" in native.last_error()
    lib.wekws_model_destroy(h)
    cfg = native.FbankConfig(16000, 300, 160, 512, 80, 0.97, 1, 1e-7)
    w = torch.ones(400)
    mel = torch.zeros(80, 256)
    assert lib.wekws_fbank_create(C.byref(cfg), C.c_void_p(w.data_ptr()), C.c_void_p(mel.data_ptr()), C.byref(h)) == -1
    assert "frame_length" in native.last_error()
    assert lib.wekws_fbank_num_frames(None, 16000) == 98
    assert lib.wekws_fbank_num_frames(None, 399) == 0


@pytest.mark.parametrize("case", CASE_NAMES)
def test_fold_and_pack_reproduce_the_oracle(case, native):
    cfg, model, B = build_model(case, init_model)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    h = model._build_handle(finalize=False)          # host-only half of finalize
    stream, vec = PE.read_packed(native, h)
    bb = cfg["backbone"]
    has_cmvn = model.global_cmvn is not None
    sig = "activation" not in cfg
    x = synth.features(B, 21, cfg["input_dim"], seed=3, cmvn_like=has_cmvn)
    if bb["type"] == "gru":
        h0 = torch.randn(bb["num_layers"], B, cfg["hidden_dim"], generator=torch.Generator().manual_seed(1))
        y_ref, c_ref = O.kws_forward(sd, cfg, x, h0)
        y, c = PE.eval_gru(vec, cfg["hidden_dim"], bb["num_layers"], cfg["input_dim"], cfg["output_dim"], sig,
                           has_cmvn, x, h0)
    else:
        kind = "mdtc" if bb["type"] == "mdtc" else ("ds_tcn" if bb.get("ds") else "tcn")
        K = bb.get("kernel_size", 8)
        dils = [1] + [2 ** l for _ in range(bb["num_stack"]) for l in range(bb["stack_size"])] \
            if kind == "mdtc" else [2 ** i for i in range(bb["num_layers"])]
        P = model.backbone.padding
        cache = torch.randn(B, model.hdim, P, generator=torch.Generator().manual_seed(2))
        y_ref, c_ref = O.kws_forward(sd, cfg, x, cache)
        y, c = PE.eval_conv(stream, vec, kind, model.hdim, cfg["input_dim"], cfg["output_dim"], K, dils,
                            bb.get("stack_size", 1), sig, has_cmvn, x, cache)
    assert (y - y_ref).abs().max() <= 2e-5 * max(1.0, float(y_ref.abs().max()))
    assert (c - c_ref).abs().max() <= 2e-5 * max(1.0, float(c_ref.abs().max()))


@pytest.mark.parametrize("name", ["mdtc", "tcn", "ds_tcn"])
def test_tensor_core_weight_images_encode_the_folded_gemms(name, native):
    """The pre-swizzled bf16 hi|lo images the tcgen05 kernels read (K-major SWIZZLE_128B, tc_common.cuh) decode back
    to the folded FP32 GEMM matrices of the FP32 path: hi = bf16_rn(w), |hi + lo - w| <= 2^-16 |w|, zero padding
    beyond K.  Pins write_w_image / write_w_image128 and the image order without a GPU."""
    import ctypes as C
    import numpy as np
    cfg = model_config(name)
    model = synth.randomize_(init_model(cfg)).eval()
    h = model._build_handle(finalize=False)
    stream, _ = PE.read_packed(native, h)
    lib = native.lib()
    n = lib.wekws_model_packed_floats(h, 2)
    assert n > 0, "no tensor-core images packed"
    raw = torch.empty(n, dtype=torch.float32)
    native.check(lib.wekws_model_packed_copy(h, 2, C.c_void_p(raw.data_ptr()), n), "packed_copy")
    img = raw.numpy().view(np.uint16)
    Cc, idim = model.hdim, cfg["input_dim"]
    K = cfg["backbone"].get("kernel_size", 8)
    nblk = 17 if name == "mdtc" else 4
    # FP32 stream: W^T [K][C] matrices in consumption order
    mats, pos = [], 0

    def take(rows):
        nonlocal pos
        w = stream[pos:pos + rows * Cc].reshape(rows, Cc).numpy()
        pos += rows * Cc
        return w
    mats.append(take(idim))
    per_block = {"mdtc": 2, "tcn": K, "ds_tcn": 1}[name]
    for _ in range(nblk * per_block):
        mats.append(take(Cc))
    assert pos == stream.numel()

    def decode(off_u16, rows):                       # -> (hi, lo) float arrays [rows][64] of one image
        nn, kk = np.meshgrid(np.arange(rows), np.arange(64), indexing="ij")
        byte = nn * 128 + (((kk >> 3) ^ (nn & 7)) << 4) + (kk & 7) * 2
        def f(u):
            return (u.astype(np.uint32) << 16).view(np.float32)
        return f(img[off_u16 + byte // 2]), f(img[off_u16 + rows * 64 + byte // 2])

    def check(hi, lo, w):                            # w [rows_n][64 k] (zero where k >= K of the matrix)
        rn = torch.from_numpy(w.copy()).to(torch.bfloat16).float().numpy()
        assert np.array_equal(hi, rn)
        assert np.all(np.abs(hi + lo - w) <= 2.0 ** -16 * np.abs(w) + 1e-30)

    def slab(m, k0, n0, rows):                       # W^T [K][C] -> [n][k] block, zero padded in k
        out = np.zeros((rows, 64), np.float32)
        kend = min(k0 + 64, m.shape[0])
        if kend > k0:
            out[:, :kend - k0] = m[k0:kend, n0:n0 + rows].T
        return out

    u = 0
    if name == "ds_tcn":
        plan = [(0, 64 * a, 128 * hh) for a in range((idim + 63) // 64) for hh in range(2)]
        plan += [(1 + b, 64 * ks, 128 * hh) for b in range(nblk) for ks in range(4) for hh in range(2)]
        rows = 128
    else:
        plan = [(0, 0, 0), (0, 64, 0)] + [(1 + g, 0, 0) for g in range(nblk * per_block)]
        rows = 64
    for mi, k0, n0 in plan:
        hi, lo = decode(u, rows)
        check(hi, lo, slab(mats[mi], k0, n0, rows))
        u += rows * 64 * 2
    assert u == img.size


@pytest.mark.parametrize("idim,layers", [(80, 2), (40, 1)])
def test_gru_tensor_core_weight_stream_encodes_the_gate_matrices(idim, layers, native):
    """The per-step weight stream of the tensor-core GRU kernel (gru_tc.cu: 16 KB K-major SWIZZLE_128B bf16 chunks of
    128 hidden units x 64 K, hi chunk then lo chunk per K slab, in the order the MMA issuer consumes them: Linear, then
    per layer W_hh (r, z, n) and W_ih (r, z, n)) decodes back to the module's own weight matrices."""
    import ctypes as C
    import numpy as np
    cfg = model_config("gru", input_dim=idim)
    cfg["backbone"]["num_layers"] = layers
    model = synth.randomize_(init_model(cfg)).eval()
    h = model._build_handle(finalize=False)
    lib = native.lib()
    n = lib.wekws_model_packed_floats(h, 2)
    nchunk = 2 * ((idim + 63) // 64) + 24 * layers
    assert n * 4 == nchunk * 16384
    raw = torch.empty(n, dtype=torch.float32)
    native.check(lib.wekws_model_packed_copy(h, 2, C.c_void_p(raw.data_ptr()), n), "packed_copy")
    img = raw.numpy().view(np.uint16)
    sd = model.state_dict()
    nn, kk = np.meshgrid(np.arange(128), np.arange(64), indexing="ij")
    u16 = (nn * 128 + (((kk >> 3) ^ (nn & 7)) << 4) + (kk & 7) * 2) // 2

    def chunk(i):
        return (img[i * 8192 + u16].astype(np.uint32) << 16).view(np.float32)

    def check(i, W, row0, k0):                       # chunks i (hi), i + 1 (lo) <- W[row0:row0+128, k0:k0+64]
        w = np.zeros((128, 64), np.float32)
        kend = min(k0 + 64, W.shape[1])
        w[:, :kend - k0] = W[row0:row0 + 128, k0:kend]
        hi, lo = chunk(i), chunk(i + 1)
        assert np.array_equal(hi, torch.from_numpy(w.copy()).to(torch.bfloat16).float().numpy())
        assert np.all(np.abs(hi + lo - w) <= 2.0 ** -16 * np.abs(w) + 1e-30)

    i = 0
    wp = sd["preprocessing.out.0.weight"].numpy()
    for s in range((idim + 63) // 64):
        check(i, wp, 0, 64 * s)
        i += 2
    for layer in range(layers):
        for key in ("weight_hh", "weight_ih"):
            W = sd[f"backbone.{key}_l{layer}"].numpy()
            for g in range(3):
                for s in range(2):
                    check(i, W, 128 * g, 64 * s)
                    i += 2
    assert i == nchunk


def test_state_dict_schema_and_init_match_reference_golden():
    d = golden("init_digest")
    for name in ("mdtc", "mdtc_small", "ds_tcn", "tcn", "gru"):
        torch.manual_seed(777)
        m = init_model(model_config(name))
        assert len(m.state_dict()) == int(d[name + "_nkeys"])
        # same module construction order => same RNG stream => bit-identical initial weights
        assert abs(synth.state_digest(m) - float(d[name])) <= 1e-9 * float(d[name])
    m = init_model(model_config("mdtc"))
    assert m.backbone.padding == 244 and m.hdim == 64 and m.idim == 80 and m.odim == 1
    assert init_model(model_config("ds_tcn")).backbone.padding == 105


@pytest.mark.parametrize("name", ["mdtc", "mdtc_small", "ds_tcn", "tcn", "gru"])
def test_checkpoints_interchange_with_live_reference(name, tmp_path):
    """A checkpoint with exactly the reference's state_dict schema (key, shape, dtype of every entry its init_model
    builds for the same config: tests/golden/checkpoint_schema.npz) loads strictly, and ours has that schema."""
    g = golden("checkpoint_schema")
    dims = iter(g[name + "_dims"].tolist())
    schema = {k: (tuple(next(dims) for _ in range(nd)), dt)
              for k, nd, dt in zip(g[name + "_keys"].tolist(), g[name + "_ndim"].tolist(), g[name + "_dtypes"].tolist())}
    gen = torch.Generator().manual_seed(5)
    ref_sd = {k: (torch.full(shape, 100, dtype=getattr(torch, dt)) if dt == "int64"
                  else torch.randn(shape, generator=gen).to(getattr(torch, dt)))
              for k, (shape, dt) in schema.items()}
    ours = init_model(model_config(name))
    path = str(tmp_path / "ckpt.pt")
    torch.save(ref_sd, path)                                # utils/checkpoint.py:46-50
    missing = ours.load_state_dict(torch.load(path), strict=True)   # utils/checkpoint.py:30
    assert not missing.missing_keys and not missing.unexpected_keys
    assert all(torch.equal(v, ref_sd[k]) for k, v in ours.state_dict().items())
    # what the reference's own strict load of our state_dict checks (keys, shapes), and the dtypes
    assert {k: (tuple(v.shape), str(v.dtype).replace("torch.", "")) for k, v in ours.state_dict().items()} == schema
    # average_model.py:77-83 turns num_batches_tracked into float: loading must still work
    avg = {k: (v.float() if v.dtype == torch.int64 else v) for k, v in ref_sd.items()}
    ours.load_state_dict(avg, strict=True)


def test_unsupported_configs_and_cpu_inputs_fail_loudly():
    with pytest.raises(NotImplementedError):
        init_model(dict(model_config("mdtc"), preprocessing=dict(type="cnn1d_s1")))
    with pytest.raises(NotImplementedError):
        init_model(dict(model_config("mdtc"), classifier=dict(type="global", dropout=0.5)))
    with pytest.raises(SystemExit):                         # kws_model.py:124-125 behaviour
        init_model(dict(model_config("mdtc"), preprocessing=dict(type="bogus")))
    m = init_model(model_config("mdtc"))
    with pytest.raises(RuntimeError, match="eval"):
        m(torch.zeros(1, 4, 80))
    m.eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 4, 80))
    with pytest.raises(RuntimeError, match="CUDA"):
        Fbank(80)(torch.zeros(1, 16000))


def test_frontend_constants_are_the_reference_tables():
    g = golden("fbank")
    assert np.array_equal(frontend.window_function("povey", 400).numpy(), g["povey_window"])
    for nmel in (80, 40):
        assert np.array_equal(frontend.mel_filterbank(nmel, 512, 16000.0).numpy(), g[f"mel{nmel}"])
    mel = frontend.mel_filterbank(80, 512, 16000.0)
    assert int((mel != 0).sum()) == 501 and int((mel != 0).sum(1).max()) <= 16      # SURVEY 8a F4
    fb = Fbank(80)
    assert fb.num_frames(16000) == 98 and fb.num_frames(399) == 0 and fb.num_frames(400) == 1
    assert fb.n_fft == 512 and fb.win == 400 and fb.shift == 160


def test_cmvn_loaders(tmp_path):
    from wekws_b200 import load_cmvn, load_kaldi_cmvn
    p = synth.write_cmvn_json(80, seed=7, path=str(tmp_path / "c.json"))
    assert np.array_equal(load_cmvn(p), golden("cmvn")["cmvn"])
    k = tmp_path / "kaldi_cmvn.txt"
    k.write_text("<Nnet>\n<Splice> 6 2\n[ 0 1 2 ]\n<AddShift> 2 2\n<LearnRateCoef> 0 [ -1.5 -2.5 ]\n"
                 "<Rescale> 2 2\n<LearnRateCoef> 0 [ 0.5 0.25 ]\n</Nnet>\n")
    out = load_kaldi_cmvn(str(k))
    assert out.shape == (2, 6) and np.allclose(out[0, :2], [1.5, 2.5]) and np.allclose(out[1, :2], [0.5, 0.25])


def test_patch_reference_rebinds_the_reference_factory(tmp_path):
    """patch_reference() (wekws_b200/overlay.py): with the reference importable, `wekws.model.kws_model.init_model`
    and `.KWSModel` -- the names wekws/bin/score.py:30 and average_model / stream_kws_ctc import -- become this
    implementation; without it a stub package of the same dotted name is registered.  The importable reference is
    stood in for by a package of the same dotted names written to tmp_path.  Run in subprocesses so the rest of this
    session keeps the unpatched modules."""
    import subprocess
    import sys
    code_stub = ("import sys; sys.path.insert(0, %r)\n"
                 "from wekws_b200 import patch_reference; import wekws_b200.kws_model as ours\n"
                 "assert patch_reference() is False\n"
                 "from wekws.model.kws_model import init_model, KWSModel\n"
                 "assert init_model is ours.init_model and KWSModel is ours.KWSModel\n" % ROOT)
    r = subprocess.run([sys.executable, "-c", code_stub], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    model_dir = tmp_path / "wekws" / "model"
    model_dir.mkdir(parents=True)
    (tmp_path / "wekws" / "__init__.py").write_text("")
    (model_dir / "__init__.py").write_text("")
    (model_dir / "kws_model.py").write_text("class KWSModel:\n    pass\n\n\ndef init_model(configs):\n"
                                            "    return KWSModel()\n")
    (model_dir / "mdtc.py").write_text("")
    code_real = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
                 "import wekws.model.kws_model as ref; orig = ref.init_model\n"
                 "from wekws_b200 import patch_reference; import wekws_b200.kws_model as ours\n"
                 "assert patch_reference() is True\n"
                 "from wekws.model.kws_model import init_model, KWSModel\n"
                 "assert init_model is ours.init_model and init_model is not orig and KWSModel is ours.KWSModel\n"
                 "import wekws.model.mdtc  # the rest of the reference package stays importable\n"
                 % (ROOT, str(tmp_path)))
    r = subprocess.run([sys.executable, "-c", code_real], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
