"""Pins the CPU oracle (oracle/kws_oracle.py) to the reference: golden vectors produced by the
real reference (oracle/make_golden.py, oracle/make_reference_golden.py)."""
import numpy as np
import pytest
import torch

from oracle import kws_oracle as O
from tests.cases import CASE_NAMES, CHUNKS, build_model
from tests.conftest import golden
from wekws_b200 import init_model, synth

TOL_MODEL = 2e-6      # oracle uses the same ATen ops as the reference: agreement is ~1 ulp
TOL_FBANK = 2e-5      # same ops (rfft, mm) -- identical up to thread-count dependent summation order


def _oracle_model(case):
    # weights come from the product's holder modules (same state_dict schema as the reference);
    # the digest check proves they are the weights the golden was generated with
    cfg, model, B = build_model(case, init_model)
    return cfg, {k: v.clone() for k, v in model.state_dict().items()}, model, B


@pytest.mark.parametrize("case", CASE_NAMES)
def test_oracle_matches_reference_golden(case):
    g = golden("model_" + case)
    cfg, sd, model, B = _oracle_model(case)
    assert abs(synth.state_digest(model) - float(g["digest"])) < 1e-6 * float(g["digest"])
    assert sorted(sd.keys()) == list(g["keys"])
    gru = cfg["backbone"]["type"] == "gru"
    cache = torch.zeros(cfg["backbone"]["num_layers"], B, cfg["hidden_dim"]) if gru else None
    for i, T in enumerate(CHUNKS):
        x = torch.from_numpy(g[f"x{i}"])
        assert x.shape[1] == T
        y, cache = O.kws_forward(sd, cfg, x, cache)
        assert np.abs(y.numpy() - g[f"y{i}"]).max() <= TOL_MODEL * max(1.0, np.abs(g[f"y{i}"]).max())
        if f"c{i}" in g:
            assert np.abs(cache.numpy() - g[f"c{i}"]).max() <= 1e-5
    full = torch.cat([torch.from_numpy(g[f"x{i}"]) for i in range(len(CHUNKS))], dim=1)
    c0 = torch.zeros(cfg["backbone"]["num_layers"], B, cfg["hidden_dim"]) if gru else None
    yf, _ = O.kws_forward(sd, cfg, full, c0)
    assert np.abs(yf.numpy() - g["y_full"]).max() <= TOL_MODEL * max(1.0, np.abs(g["y_full"]).max())


def test_oracle_fbank_matches_reference_golden():
    g = golden("fbank")
    names = [k[4:] for k in g.files if k.startswith("wav_")]
    assert len(names) >= 9
    for name in names:
        wav = torch.from_numpy(g["wav_" + name])
        for nmel in (80, 40):
            ref = g[f"fbank{nmel}_{name}"]
            out = O.fbank(wav, num_mel_bins=nmel).numpy()
            assert out.shape == ref.shape, name
            if ref.size:
                assert np.abs(out - ref).max() <= TOL_FBANK, (name, nmel, np.abs(out - ref).max())
    ham = O.fbank(torch.from_numpy(g["wav_gauss3000_a"]), window_type="hamming").numpy()
    assert np.abs(ham - g["fbank80_hamming_gauss3000_a"]).max() <= TOL_FBANK
    # all-zero audio gives exactly log(eps) in every bin (SURVEY 8c)
    z = O.fbank(torch.zeros(1200)).numpy()
    assert np.all(z == np.float32(np.log(np.float32(O.EPS))))


@pytest.mark.parametrize("case", ["fsmn", "fsmn_strided"])
def test_oracle_fsmn_matches_reference_golden(case):
    """SURVEY 8f-4 groundwork: the FSMN restatement against the real reference (weights travel in the golden file)."""
    from tests.cases import fsmn_config
    g = golden("model_" + case)
    cfg = fsmn_config(case)
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd_")}
    cache, i = None, 0
    while f"x{i}" in g.files:
        y, cache = O.kws_forward(sd, cfg, torch.from_numpy(g[f"x{i}"]), cache)
        assert np.abs(y.numpy() - g[f"y{i}"]).max() <= TOL_MODEL * max(1.0, np.abs(g[f"y{i}"]).max()), (case, i)
        assert cache.shape == g[f"c{i}"].shape and np.abs(cache.numpy() - g[f"c{i}"]).max() <= 1e-5
        i += 1
    assert i == 4
    # streaming == whole utterance (the right context only delays the output, fsmn.py:238-248)
    full = torch.cat([torch.from_numpy(g[f"x{j}"]) for j in range(i)], dim=1)
    yf, _ = O.kws_forward(sd, cfg, full, None)
    assert np.abs(yf.numpy() - g["y_full"]).max() <= TOL_MODEL * max(1.0, np.abs(g["y_full"]).max())


def test_oracle_mfcc_matches_reference_golden():
    """kaldi.mfcc as wekws/dataset/processor.py:157-166 calls it (fixtures from oracle/make_golden.py gen_mfcc)."""
    g, fb = golden("mfcc"), golden("fbank")
    keys = [k for k in g.files if k.startswith("mfcc")]
    assert len(keys) >= 18
    for k in keys:
        head, nmel, name = k.split("_", 2)
        nc, nmel = int(head[4:]), int(nmel)
        out = O.mfcc(torch.from_numpy(fb["wav_" + name]), nc, nmel).numpy()
        assert out.shape == g[k].shape, k
        # same ops as torchaudio (fbank -> matmul -> lifter); the matmul's summation order depends on the BLAS thread count
        assert np.abs(out - g[k]).max() <= 2e-4, (k, np.abs(out - g[k]).max())
    assert np.array_equal(O.dct_matrix(80, 80).numpy(), g["dct80"])
    assert np.array_equal(O.dct_matrix(13, 23).numpy(), g["dct13_23"])
    assert O.mfcc(torch.zeros(399)).shape == (0, 80)


def test_oracle_cmvn_loader_matches_golden(tmp_path):
    p = synth.write_cmvn_json(80, seed=7, path=str(tmp_path / "cmvn.json"))
    mean, istd = O.load_cmvn_json(p)
    ref = golden("cmvn")["cmvn"]
    assert np.allclose(mean.numpy(), ref[0].astype(np.float32), rtol=0, atol=0)
    assert np.allclose(istd.numpy(), ref[1].astype(np.float32), rtol=0, atol=0)


@pytest.mark.parametrize("case", CASE_NAMES)
def test_oracle_matches_live_reference(case):
    """The same input streamed three times in 23-frame chunks, cache carried, against what the reference's own
    KWSModel returned (tests/golden/stream23.npz: every output, the cache at a fixed sample of its live entries)."""
    g = golden("stream23")
    cfg, sd, model, B = _oracle_model(case)
    assert abs(synth.state_digest(model) - float(g[case + "_digest"])) < 1e-6 * float(g[case + "_digest"])
    gru = cfg["backbone"]["type"] == "gru"
    x = synth.features(B, 23, cfg["input_dim"], seed=5, cmvn_like=model.global_cmvn is not None)
    assert abs(float(x.double().sum()) - float(g[case + "_x_sum"])) <= 1e-9 * float(x.double().abs().sum())
    c_or = torch.zeros(cfg["backbone"]["num_layers"], B, cfg["hidden_dim"]) if gru else None
    idx = torch.from_numpy(g[case + "_cidx"])
    for i in range(3):
        y_ref, c_ref = torch.from_numpy(g[f"{case}_y{i}"]), torch.from_numpy(g[f"{case}_c{i}"])
        y_or, c_or = O.kws_forward(sd, cfg, x, c_or)
        assert y_or.shape == y_ref.shape and tuple(c_or.shape) == tuple(g[case + "_cshape"])
        assert (y_ref - y_or).abs().max() <= TOL_MODEL * max(1.0, float(y_ref.abs().max()))
        assert (c_ref - c_or.reshape(-1)[idx]).abs().max() <= 1e-5


def _sampled_frames(g, name):
    return tuple(g[name + "_shape"]), torch.from_numpy(g[name + "_frames"]), torch.from_numpy(g[name])


def test_oracle_mfcc_matches_live_torchaudio():
    """Against torchaudio.compliance.kaldi.mfcc on the same audio (tests/golden/kaldi_live.npz, a fixed sample of
    40 frames)."""
    pcm = synth.pcm_int16(1, 16000 * 2, seed=78)[0].float()
    shape, frames, ref = _sampled_frames(golden("kaldi_live"), "mfcc80_seed78")
    out = O.mfcc(pcm)
    assert tuple(out.shape) == shape
    assert (out[frames] - ref).abs().max() <= 2e-4


def test_oracle_fbank_matches_live_torchaudio():
    """Against torchaudio.compliance.kaldi.fbank on the same audio (tests/golden/kaldi_live.npz, a fixed sample of
    40 frames)."""
    pcm = synth.pcm_int16(1, 16000 * 3, seed=77)[0].float()
    shape, frames, ref = _sampled_frames(golden("kaldi_live"), "fbank80_seed77")
    out = O.fbank(pcm)
    assert tuple(out.shape) == shape
    assert (out[frames] - ref).abs().max() <= TOL_FBANK


def test_oracle_det_stats_pinned_to_reference_compute_det():
    """O.det_stats + O.det_curve_text == the stats files the REFERENCE's wekws/bin/compute_det.py wrote for the same
    score / label files (tests/golden/det_stats.npz, made by oracle/make_det_golden.py), byte for byte."""
    g = golden("det_stats")
    post, lens = torch.from_numpy(g["post"]), torch.from_numpy(g["lens"])
    kinds, durs = g["kinds"].tolist(), g["durations"].tolist()
    for si, (ws, step) in enumerate(g["settings"].tolist()):
        thr, ms, tr = O.det_stats(post, lens, step, int(ws))
        for k in range(post.shape[2]):
            assert O.det_curve_text(thr, ms, tr, kinds, durs, k) == str(g[f"stats_{si}_{k}"]), (si, k)


def test_oracle_context_expansion_pinned_to_reference_processor():
    """O.context_expansion / O.frame_skip == the reference's own processor functions (tests/golden/context.npz, made by
    oracle/make_context_golden.py running wekws/dataset/processor.py:267-312), bit for bit."""
    g = golden("context")
    for i, (T, D, left, right, skip) in enumerate(g["cases"].tolist()):
        y = O.frame_skip(O.context_expansion(torch.from_numpy(g[f"x{i}"]), left, right), skip)
        assert torch.equal(y, torch.from_numpy(g[f"y{i}"])), i


def _ctc_golden_cases():
    g = golden("ctc")
    tokenset = set(g["tokenset"].tolist())
    for i in range(int(g["ncases"])):
        n = int(g[f"n{i}"])
        hyps = []
        for k in range(n):
            ln = int(g[f"len{i}"][k])
            hyps.append((tuple(g[f"tok{i}"][k, :ln].tolist()), float(g[f"score{i}"][k]),
                         [dict(token=int(g[f"tok{i}"][k, j]), frame=int(g[f"frame{i}"][k, j]), prob=float(g[f"prob{i}"][k, j]))
                          for j in range(ln)]))
        yield i, torch.from_numpy(g[f"probs{i}"]), (tokenset if bool(g[f"use_set{i}"]) else None), hyps


def test_oracle_ctc_prefix_beam_search_pinned_to_reference():
    """O.ctc_prefix_beam_search == the hypotheses the REFERENCE's wekws/model/loss.py:206-312 returned for the same
    posteriors (tests/golden/ctc.npz, made by oracle/make_ctc_golden.py): order, prefixes, scores (double, exact),
    node frames and probabilities; chunked decoding with carried hypotheses == whole utterance."""
    for i, probs, tokenset, want in _ctc_golden_cases():
        got = O.hyps_of(O.ctc_prefix_beam_search(probs, tokenset))
        assert got == want, i
        cur = None
        for t0 in range(0, probs.size(0), 17):
            cur = O.ctc_prefix_beam_search(probs[t0:t0 + 17], tokenset, cur_hyps=cur, frame_offset=t0)
        assert O.hyps_of(cur) == want, i
