"""CTC test-set scoring (wekws_b200.ctc_stream_score, csrc/ctc_score.cu) and DET statistics (compute_det_ctc) against
the reference's stream_score_ctc.py / score_ctc.py / compute_det_ctc.py: the CPU oracle (oracle/ctc_score_oracle.py)
is pinned to what the reference scripts wrote (tests/golden/ctc_score.npz); the device is checked against the golden
text and the oracle, byte for byte."""
import io
import json
import os

import numpy as np
import pytest
import torch

from oracle import ctc_score_oracle as SO
from oracle import kws_oracle as O
from tests.conftest import golden
from wekws_b200 import ctc_score as CS


def _keywords(spec, char_ids):
    """{keyword: {'token_id': (...)}} as the scripts build it from --keywords (one token per character)."""
    return {w: {"token_id": tuple(char_ids[c] for c in w)} for w in spec.split(",")}


def _cases():
    g = golden("ctc_score")
    char_ids = json.loads(str(g["char_ids"]))
    out = []
    for ci in range(int(g["ncases"])):
        p = f"c{ci}_"
        th, mn, mx, sb, pb, fs = g[p + "flags"].tolist()
        batches = [dict(probs=torch.from_numpy(g[p + f"b{bi}_probs"]), lengths=g[p + f"b{bi}_lengths"].tolist(),
                        keys=[str(k) for k in g[p + f"b{bi}_keys"]]) for bi in range(int(g[p + "nbatches"]))]
        out.append(dict(name=str(g[p + "name"]), keywords=_keywords(str(g[p + "keywords"]), char_ids),
                        flags=dict(threshold=th, min_frames=int(mn), max_frames=int(mx), score_beam=int(sb),
                                   path_beam=int(pb), frame_skip=int(fs)),
                        batches=batches, stream_text=str(g[p + "stream_text"]),
                        score_ctc_text=str(g[p + "score_ctc_text"])))
    return out


def _det_cases():
    g = golden("ctc_score")
    out = []
    for di in range(int(g["ndet"])):
        p = f"d{di}_"
        labels = [json.loads(line) for line in str(g[p + "data_list"]).splitlines()]
        kws = str(g[p + "keywords"]).split(",")
        out.append(dict(name=str(g[p + "name"]), labels=labels, score=str(g[p + "score"]).splitlines(True),
                        true_keywords={k: k for k in kws}, step=float(g[p + "step"]),
                        stats=dict(zip([str(n) for n in g[p + "stats_names"]], [str(t) for t in g[p + "stats_texts"]]))))
    return out


def _oracle_text(case, events=None):
    f = case["flags"]
    out = []
    for bt in case["batches"]:
        for b, key in enumerate(bt["keys"]):
            out.extend(SO.stream_score(key, bt["probs"][b, :bt["lengths"][b]], case["keywords"], f["threshold"],
                                       f["min_frames"], f["max_frames"], f["score_beam"], f["path_beam"],
                                       f["frame_skip"], events)[0])
    return "".join(out)


# ----------------------------------------------------------------------------------------------------------- CPU
def test_oracle_matches_reference_score_files():
    """The oracle's stream_score_ctc.py lines == the reference's file; the whole-utterance search + look-up of
    kws_oracle == the reference's score_ctc.py file, on the same probabilities."""
    for case in _cases():
        assert _oracle_text(case) == case["stream_text"], case["name"]
        idx = {0} | {t for w in case["keywords"] for t in case["keywords"][w]["token_id"]}
        lines = []
        for bt in case["batches"]:
            for b, key in enumerate(bt["keys"]):
                hyps = O.hyps_of(O.ctc_prefix_beam_search(bt["probs"][b, :bt["lengths"][b]], idx))
                word, score, _, _ = O.ctc_keyword_hit(hyps, case["keywords"])
                lines.append(f"{key} detected {word} {score:.3f}\n" if word is not None else f"{key} rejected\n")
        assert "".join(lines) == case["score_ctc_text"], case["name"]


def test_oracle_matches_reference_stats_files():
    for case in _det_cases():
        got = SO.det_stats_text(case["labels"], case["score"], case["true_keywords"], case["step"])
        assert got == case["stats"], case["name"]


def test_golden_covers_the_cases():
    cases = {c["name"]: c for c in _cases()}
    events = {}
    for c in cases.values():
        _oracle_text(c, events)
    assert events.get("skipped", 0) > 0 and events.get("threshold_reject", 0) > 0
    assert events.get("carried_sqrt", 0) > 0 and events.get("stale_duration", 0) > 0
    texts = "".join(c["stream_text"] for c in cases.values())
    keys = [line.split()[0] for line in texts.splitlines() if " detected " in line]
    assert max(keys.count(k) for k in set(keys)) >= 2                       # several activations in one utterance
    lens = [n for c in cases.values() for bt in c["batches"] for n in bt["lengths"]]
    T = [bt["probs"].size(1) for c in cases.values() for bt in c["batches"]]
    assert 0 in lens and min(lens) < min(T)                                  # zero length, padded batches
    skips = {c["flags"]["frame_skip"] for c in cases.values()}
    assert skips == {1, 3}
    assert any(c["flags"]["score_beam"] < 3 and c["flags"]["path_beam"] < 20 for c in cases.values())
    assert any(len(set(v["token_id"])) < len(v["token_id"]) for c in cases.values() for v in c["keywords"].values())
    # the keyword order matters: reversed dict order gives another score file
    c = cases["kw_order"]
    rev = dict(c, keywords=dict(reversed(list(c["keywords"].items()))))
    assert _oracle_text(rev) != c["stream_text"]
    dets = {d["name"]: d for d in _det_cases()}
    assert {d["step"] for d in dets.values()} == {0.01, 0.001}
    mixed = dets["det_mixed"]
    assert any(any("a" <= ch <= "z" for ch in o["txt"].lower()) and any(ord(ch) > 0x3000 for ch in o["txt"])
               for o in mixed["labels"])
    assert any(" rejected" in s for s in mixed["score"])
    # keyword utterances that score -1.0 for their keyword: rejected, and detected as the other keyword
    why = set()
    for d in dets.values():
        first = {}
        for line in d["score"]:
            arr = line.split()
            first.setdefault(arr[0], arr[2] if arr[1] == "detected" else None)
        tables = SO.load_label_and_score(list(d["true_keywords"]), d["labels"], d["score"], d["true_keywords"])
        for kw, tab in tables.items():
            for key, confi in tab["keyword_table"].items():
                if confi == -1.0:
                    why.add("rejected" if first[key] is None else
                            "other" if SO.space_mixed_label(first[key]) != kw else "same")
    assert {"rejected", "other"} <= why


def _random_join_case(rng, n=300):
    kws = {"嗨小问": "嗨小问", "heysnips": "HEYSNIPS", "你好问问": "你好问问"}
    txts = ["嗨小问", "hey 嗨小问", "你好 问问", "HeySnips 你好", "今天", "heysnips!", "ok heysnips 嗨", " 嗨小问 "]
    labels = [{"key": f"k{i}", "txt": txts[int(rng.integers(len(txts)))], "duration": float(rng.uniform(0.1, 9))}
              for i in range(n)]
    lines = []
    for o in labels:
        for _ in range(int(rng.integers(1, 4))):
            r = rng.random()
            kw = list(kws)[int(rng.integers(3))]
            lines.append(f"{o['key']} rejected\n" if r < 0.25 else f"{o['key']} detected {kw} {rng.random():.3f}\n")
    rng.shuffle(lines)
    return labels, lines, kws


def test_host_join_equals_oracle_on_random_sets():
    rng = np.random.default_rng(3)
    for _ in range(20):
        labels, lines, kws = _random_join_case(rng)
        got = CS.ctc_det_tables(labels, lines, kws)
        want = SO.load_label_and_score(list(kws), labels, lines, kws)
        assert got == want
        assert list(got) == list(want)
        for k in got:                                    # durations: the same float sums, bit for bit
            assert got[k]["filler_duration"].hex() == want[k]["filler_duration"].hex()
    for text in ["HeySnips 你好", "a b c", " 嗨 x", "ab,cd 问", "\t嗨", "ÄbC 你"]:
        assert CS.space_mixed_label(text) == SO.space_mixed_label(text)
        assert CS.split_mixed_label(text) == SO.split_mixed_label(text)


def test_host_join_errors():
    labels = [{"key": "a", "txt": "嗨小问", "duration": 1.0}, {"key": "b", "txt": "x", "duration": 1.0}]
    with pytest.raises(KeyError):                        # a label key without a score line
        CS.ctc_det_tables(labels, ["a detected 嗨小问 0.5\n"], {"嗨小问": "嗨小问"})
    with pytest.raises(AssertionError):
        SO.load_label_and_score(["嗨小问"], labels, ["a detected 嗨小问 0.5\n"], {"嗨小问": "嗨小问"})
    # duplicate keys: the first score line wins in both
    lines = ["a detected 嗨小问 0.5\n", "a rejected\n", "b rejected\n", "b detected 嗨小问 0.9\n"]
    t = CS.ctc_det_tables(labels, lines, {"嗨小问": "嗨小问"})
    assert t == SO.load_label_and_score(["嗨小问"], labels, lines, {"嗨小问": "嗨小问"})
    assert t["嗨 小 问"]["keyword_table"] == {"a": 0.5} and t["嗨 小 问"]["filler_table"] == {"b": -1.0}


# ----------------------------------------------------------------------------------------------------------- GPU
def _device_text(case, max_detections=16):
    f = case["flags"]
    buf = io.StringIO()
    for bt in case["batches"]:
        probs, lens, keys = bt["probs"], bt["lengths"], bt["keys"]
        sc = CS.ctc_stream_score(probs.cuda(), lens, case["keywords"], f["threshold"], f["min_frames"],
                                 f["max_frames"], f["score_beam"], f["path_beam"], f["frame_skip"], max_detections)
        CS.write_ctc_stream_scores(buf, keys, sc)
    return buf.getvalue()


@pytest.mark.gpu
def test_device_score_file_equals_golden():
    for case in _cases():
        assert _device_text(case) == case["stream_text"], case["name"]


def _ragged_set(B, V, seed, rows=(20, 400)):
    """B ragged utterances of planted posteriors at vocabulary V (keyword tokens inside the first 48 ids)."""
    from oracle.ctc_score_oracle import plant_logits
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(rows[0], rows[1], (B,), generator=g)
    lens[::97] = 0
    T = int(lens.max())
    logits = torch.randn(B, T, V, generator=g) * 0.3
    logits[:, :, :48] = plant_logits(B, T, seed)
    return logits.softmax(2), lens


KW = {"嗨小问": {"token_id": (5, 9, 23)}, "你好问问": {"token_id": (31, 7, 23, 23)}, "问问": {"token_id": (23, 23)}}


@pytest.mark.gpu
def test_device_equals_oracle_ragged_permuted():
    """~1000 ragged utterances at V = 2599, frame_skip 3: device == oracle line for line, and a permutation of the
    batch permutes the results."""
    B, V = 1000, 2599
    probs, lens = _ragged_set(B, V, 11)
    flags = dict(threshold=0.5, min_frames=6, max_frames=90, score_beam_size=3, path_beam_size=20, frame_skip=3)
    sc = CS.ctc_stream_score(probs.cuda(), lens, KW, **flags)
    keys = [f"u{b}" for b in range(B)]
    buf = io.StringIO()
    CS.write_ctc_stream_scores(buf, keys, sc)
    got = buf.getvalue()
    want = SO.stream_score_text(keys, probs, lens, KW, threshold=0.5, min_frames=6, max_frames=90, frame_skip=3)
    assert got == want
    assert got.count("detected") > 200
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(5))
    sc2 = CS.ctc_stream_score(probs[perm].cuda(), lens[perm], KW, **flags)
    for name in ("count", "overflow"):
        assert torch.equal(getattr(sc2, name).cpu(), getattr(sc, name).cpu()[perm])
    n = sc.count.cpu()
    for name in ("keyword", "score", "start", "end"):
        a, b = getattr(sc, name).cpu()[perm], getattr(sc2, name).cpu()
        for i in range(B):
            k = min(int(n[perm[i]]), sc.max_detections)
            assert torch.equal(a[i, :k], b[i, :k])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fsmn", "ds_tcn"])
def test_end_to_end_pcm_to_score_file(name):
    """PCM -> Fbank -> context_expansion -> model.forward_softmax -> ctc_stream_score: the score file == the oracle
    decode of the same device probabilities."""
    from tests.test_kws_stream import _peaky_model
    from wekws_b200 import Fbank, context_expansion, synth
    mel, ctx, skip = (80, (2, 2), 3) if name == "fsmn" else (40, None, 1)
    B = 12
    n = torch.randint(16000, 16000 * 4, (B,), generator=torch.Generator().manual_seed(2))
    pcm = synth.pcm_int16(B, int(n.max()), seed=8)
    feats = Fbank(mel)(pcm.cuda())
    flen = torch.tensor([O.num_frames(int(v)) for v in n], dtype=torch.int32)
    if ctx is not None:
        feats, flen = context_expansion(feats, ctx[0], ctx[1], skip, lengths=flen)
    cfg, model = _peaky_model(name, 11, feats[:1, :int(flen[0])].cpu())
    model = model.cuda()
    with torch.no_grad():
        probs, _ = model.forward_softmax(feats)
    kw = {"hi": {"token_id": (5, 9, 17, 23)}, "nihao": {"token_id": (31, 7, 23, 23)}}
    sc = CS.ctc_stream_score(probs.float().contiguous(), flen, kw, 0.05, 2, 100, frame_skip=skip)
    keys = [f"e{b}" for b in range(B)]
    buf = io.StringIO()
    CS.write_ctc_stream_scores(buf, keys, sc)
    p = probs.float().cpu()
    want = SO.stream_score_text(keys, p, flen, kw, threshold=0.05, min_frames=2, max_frames=100, frame_skip=skip)
    assert buf.getvalue() == want


@pytest.mark.gpu
def test_overflow_and_max_detections_make_the_writer_raise():
    T, V = 150, 48
    bad = torch.full((T, V), 1e-4)
    for t in range(T):
        bad[t, 5 if t % 2 == 0 else 9] = 1.0                                # 5 9 5 9 ...: the prefix grows every frame
    bad = bad / bad.sum(1, keepdim=True)
    probs, lens = _ragged_set(3, V, 4, rows=(100, 150))
    probs = probs[:, :T] if probs.size(1) >= T else torch.cat([probs, probs.new_zeros(3, T - probs.size(1), V)], 1)
    batch = torch.cat([probs, bad.unsqueeze(0)]).cuda()
    lens = torch.cat([lens.clamp(max=T), torch.tensor([T])])
    sc = CS.ctc_stream_score(batch, lens, KW, 0.0, 2, 250, frame_skip=1)
    ov = sc.overflow.cpu().tolist()
    assert ov[3] == 1 and ov[:3] == [0, 0, 0]
    with pytest.raises(RuntimeError, match="u3"):
        CS.write_ctc_stream_scores(io.StringIO(), ["u0", "u1", "u2", "u3"], sc)
    # max_detections: the count stays exact, the writer refuses to drop lines
    full = CS.ctc_stream_score(batch[:3], lens[:3], KW, 0.0, 2, 250, frame_skip=1, max_detections=16)
    counts = full.count.cpu()
    assert int(counts.max()) >= 2
    small = CS.ctc_stream_score(batch[:3], lens[:3], KW, 0.0, 2, 250, frame_skip=1, max_detections=1)
    assert torch.equal(small.count.cpu(), counts)
    assert torch.equal(small.score.cpu()[:, 0][counts > 0], full.score.cpu()[:, 0][counts > 0])
    with pytest.raises(RuntimeError, match="max_detections"):
        CS.write_ctc_stream_scores(io.StringIO(), ["u0", "u1", "u2"], small)


@pytest.mark.gpu
def test_det_sweep_equals_oracle_large():
    """~200k confidences at step 0.001, with values read back from '{:.3f}' text that sit on or next to the
    accumulated thresholds (0.3 against 0.1 + 0.1 + 0.1)."""
    from wekws_b200 import det_thresholds
    rng = np.random.default_rng(0)
    thr = det_thresholds(0.001)
    near = np.concatenate([thr.numpy(), np.nextafter(thr.numpy(), 2), np.nextafter(thr.numpy(), -1)])
    text = [float(f"{v:.3f}") for v in rng.random(60000)]
    kw = np.concatenate([rng.random(40000), text[:30000], near[:3000], [-1.0] * 2000])
    fl = np.concatenate([rng.random(90000), text[30000:], near, [-1.0] * 5000])
    assert len(kw) + len(fl) > 195000
    fr, fa = CS.ctc_det_sweep(torch.from_numpy(kw).cuda(), torch.from_numpy(fl).cuda(), thr.cuda())
    ks, fs = np.sort(kw), np.sort(fl)
    t = thr.numpy()
    assert np.array_equal(fr.cpu().numpy(), np.searchsorted(ks, t, side="left"))
    assert np.array_equal(fa.cpu().numpy(), len(fs) - np.searchsorted(fs, t, side="left"))
    assert 0.1 + 0.1 + 0.1 != 0.3 and 0.3 in set(text)
    # a direct Python count on a few thresholds, the reference's comparisons
    for i in (0, 300, 301, 700, len(t) - 1):
        assert int(fr[i]) == sum(1 for c in kw if c < t[i]) and int(fa[i]) == sum(1 for c in fl if c >= t[i])


@pytest.mark.gpu
def test_compute_det_ctc_stats_equal_golden(tmp_path):
    from wekws_b200 import compute_det_ctc
    for case in _det_cases():
        d = tmp_path / case["name"]
        d.mkdir()
        rows = compute_det_ctc(case["labels"], case["score"], case["true_keywords"], case["step"], stats_dir=str(d))
        files = {f: (d / f).read_text(encoding="utf8") for f in os.listdir(d)}
        assert files == case["stats"], case["name"]
        assert len(rows) == len(case["stats"])


@pytest.mark.gpu
def test_launch_counts():
    from wekws_b200 import _native, compute_det_ctc
    case = _cases()[0]
    bt = case["batches"][0]
    probs = bt["probs"].cuda()
    CS.ctc_stream_score(probs, bt["lengths"], case["keywords"])
    torch.cuda.synchronize()
    n0 = _native.launch_count()
    CS.ctc_stream_score(probs, bt["lengths"], case["keywords"])
    torch.cuda.synchronize()
    assert _native.launch_count() - n0 == 1
    det = _det_cases()[2]
    n0 = _native.launch_count()
    compute_det_ctc(det["labels"], det["score"], det["true_keywords"], det["step"])
    assert _native.launch_count() - n0 == len(det["true_keywords"])
