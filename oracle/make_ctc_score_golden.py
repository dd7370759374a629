#!/usr/bin/env python
"""Golden vectors for CTC test-set scoring and its DET statistics (test infrastructure): drives the REFERENCE's own
wekws/bin/stream_score_ctc.py main(), wekws/bin/score_ctc.py main() and wekws/bin/compute_det_ctc.py (run as
__main__) and stores what they wrote in tests/golden/ctc_score.npz.

    python oracle/make_ctc_score_golden.py [REFERENCE_CHECKOUT]      (default /root/reference)

Stubbed, because the scripts read files and packages that are not part of this project:
  * wenet.text.char_tokenizer.CharTokenizer -- tokenize() returns this script's fixed (strs, ids) per character;
  * wekws.dataset.init_dataset.init_dataset -- returns prepared batch dicts (keys, feats, target, lengths);
  * DataLoader                               -- identity;
  * init_model / load_checkpoint             -- a stub model that returns planted logits for the batch;
  * torch.cuda.set_device                    -- no-op (the scripts run on the CPU here);
  * matplotlib.pyplot, pypinyin.lazy_pinyin  -- no-ops (compute_det_ctc.py plots after writing the stats files).
Stored per scoring case: the float32 probabilities the reference decoded (the same logits.softmax(2) call on the same
logits), the lengths, keys and flags, and the text of both score files; per DET case: data.list, the score file, the
keywords, the step and the text of every stats file.  A rerun writes the same bytes (fixed zip timestamps).
"""
import json
import logging
import os
import runpy
import sys
import tempfile
import types

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
sys.path.insert(0, ROOT)
from oracle.ctc_score_oracle import PLANT_V as V, plant_logits  # noqa: E402
from oracle.make_kws_stream_golden import save_npz  # noqa: E402

CHAR_IDS = {"嗨": 5, "小": 9, "问": 23, "你": 31, "好": 7}      # keyword characters -> token ids
TRANSCRIPTS = ["嗨小问", "嗨 小 问", "hey 嗨小问 there", "你好问问", "你好 问问 OK", "今天天气", "HeySnips 你好",
               "嗨小", "问问", "hello world", "你好问问嗨小问", "heysnips", "ok heysnips 嗨"]

# scoring cases: flags of stream_score_ctc.py, batches (B, T), seed; case 0 has a zero-length utterance
CASES = [
    dict(name="gates_skip3", keywords="嗨小问,你好问问", frame_skip=3, threshold=0.55, min_frames=9, max_frames=45,
         score_beam=3, path_beam=20, batches=[(7, 260), (5, 200)], seed=21),
    dict(name="beams_skip1", keywords="你好问问,嗨小问", frame_skip=1, threshold=0.45, min_frames=4, max_frames=14,
         score_beam=2, path_beam=6, batches=[(6, 240)], seed=22),
    dict(name="kw_order", keywords="问问,你好问问,嗨小问", frame_skip=1, threshold=0.0, min_frames=2, max_frames=250,
         score_beam=3, path_beam=20, batches=[(6, 220)], seed=23),
]


def stub_modules(batches_box, model_box):
    for name in ["wenet", "wenet.text", "wenet.text.char_tokenizer", "wekws.dataset.init_dataset", "matplotlib",
                 "matplotlib.pyplot", "pypinyin"]:
        sys.modules[name] = types.ModuleType(name)

    class Tokenizer:
        def __init__(self, *a, **k):
            pass

        def tokenize(self, text):
            strs = text.split(" ")
            return strs, [CHAR_IDS.get(c, 1) for c in strs]

    sys.modules["wenet.text.char_tokenizer"].CharTokenizer = Tokenizer
    sys.modules["wekws.dataset.init_dataset"].init_dataset = lambda **k: batches_box[0]
    plt = sys.modules["matplotlib.pyplot"]
    for f in ["figure", "plot", "xlim", "ylim", "xticks", "yticks", "xlabel", "ylabel", "grid", "legend", "savefig"]:
        setattr(plt, f, lambda *a, **k: None)
    plt.rcParams = {}
    sys.modules["matplotlib"].pyplot = plt
    sys.modules["pypinyin"].lazy_pinyin = lambda s: [s]
    torch.cuda.set_device = lambda *a: None

    class StubModel(torch.nn.Module):
        def forward(self, feats):                      # feats[0, 0, 0] = batch index
            return model_box[int(feats[0, 0, 0])], None

    stub = StubModel()
    sys.path.insert(0, REF)
    from wekws.bin import score_ctc, stream_score_ctc     # noqa: E402  the reference's own modules
    for mod in (score_ctc, stream_score_ctc):
        mod.init_model = lambda conf: stub
        mod.load_checkpoint = lambda m, p: None
        mod.DataLoader = lambda ds, **k: ds
    return score_ctc, stream_score_ctc


def escaped(keywords):
    """The recipes pass the keywords as \\uXXXX escapes: the scripts decode them with 'unicode_escape'."""
    return keywords.encode("unicode_escape").decode("ascii")


def run_main(mod, argv):
    sys.argv = argv
    mod.main()
    logging.getLogger().handlers.clear()


def main():
    logging.disable(logging.CRITICAL)
    batches_box, model_box = [None], []
    score_ctc, stream_score_ctc = stub_modules(batches_box, model_box)
    tmp = tempfile.mkdtemp()
    out = {"V": np.array(V), "ncases": np.array(len(CASES)),
           "char_ids": np.array(json.dumps(CHAR_IDS, ensure_ascii=False))}
    labels, all_stream, all_score = [], [], []
    rng = np.random.default_rng(7)
    for ci, case in enumerate(CASES):
        batches, logits_all = [], []
        model_box.clear()
        for bi, (B, T) in enumerate(case["batches"]):
            logits = plant_logits(B, T, case["seed"] * 10 + bi)
            lens = [T] + [int(v) for v in rng.integers(T // 3, T + 1, B - 1)]
            if ci == 0 and bi == 0:
                lens[2] = 0
            keys = [f"{case['name']}_{bi}_{b}" for b in range(B)]
            model_box.append(logits)
            batches.append({"keys": keys, "feats": torch.full((B, T, 1), float(bi)),
                            "target": torch.zeros(B, 1, dtype=torch.long),
                            "feats_lengths": torch.tensor(lens), "target_lengths": torch.ones(B, dtype=torch.long)})
            logits_all.append(logits)
            for k in keys if ci < 2 else ():        # the DET cases use the two cases with the same keywords
                labels.append({"key": k, "wav": "-", "txt": TRANSCRIPTS[int(rng.integers(len(TRANSCRIPTS)))],
                               "duration": round(float(rng.uniform(0.5, 8.0)), 3)})
        batches_box[0] = batches
        cfg = os.path.join(tmp, f"{case['name']}.yaml")
        with open(cfg, "w") as f:
            yaml.safe_dump({"dataset_conf": {"filter_conf": {}, "fbank_conf": {}, "batch_conf": {},
                                             "frame_skip": case["frame_skip"]}, "model": {}}, f)
        common = ["--config", cfg, "--test_data", "-", "--checkpoint", "-", "--keywords", escaped(case["keywords"])]
        s_stream, s_score = os.path.join(tmp, f"{ci}_stream.txt"), os.path.join(tmp, f"{ci}_score.txt")
        run_main(stream_score_ctc, ["stream_score_ctc.py"] + common + [
            "--score_file", s_stream, "--threshold", str(case["threshold"]), "--min_frames", str(case["min_frames"]),
            "--max_frames", str(case["max_frames"]), "--score_beam_size", str(case["score_beam"]),
            "--path_beam_size", str(case["path_beam"])])
        run_main(score_ctc, ["score_ctc.py"] + common + ["--score_file", s_score])
        text_stream = open(s_stream, encoding="utf8").read()
        text_score = open(s_score, encoding="utf8").read()
        if ci < 2:
            all_stream.append(text_stream)
            all_score.append(text_score)
        p = f"c{ci}_"
        out.update({p + "name": np.array(case["name"]), p + "keywords": np.array(case["keywords"]),
                    p + "flags": np.array([case["threshold"], case["min_frames"], case["max_frames"],
                                           case["score_beam"], case["path_beam"], case["frame_skip"]],
                                          dtype=np.float64),
                    p + "nbatches": np.array(len(batches)),
                    p + "stream_text": np.array(text_stream), p + "score_ctc_text": np.array(text_score)})
        for bi, bd in enumerate(batches):
            out[p + f"b{bi}_probs"] = logits_all[bi].softmax(2).numpy()     # the call the scripts make (:219)
            out[p + f"b{bi}_lengths"] = bd["feats_lengths"].numpy().astype(np.int32)
            out[p + f"b{bi}_keys"] = np.array(bd["keys"])
        print(f"{case['name']}: {text_stream.count('detected')} detections, {text_stream.count('rejected')} rejected; "
              f"score_ctc {text_score.count('detected')} detected")

    # DET cases: both scorers' files over the scoring cases' utterances, and a synthetic mixed Latin / CJK test set
    data_list = "".join(json.dumps(o, ensure_ascii=False) + "\n" for o in labels)
    det = [("det_stream", data_list, "".join(all_stream), "嗨小问,你好问问", 0.01),
           ("det_score_ctc", data_list, "".join(all_score), "嗨小问,你好问问", 0.001)]
    rng = np.random.default_rng(8)
    mixed_labels, mixed_scores = [], []
    for u in range(400):
        key = f"mixed_{u:04d}"
        mixed_labels.append({"key": key, "wav": "-", "txt": TRANSCRIPTS[int(rng.integers(len(TRANSCRIPTS)))],
                             "duration": float(rng.uniform(0.3, 9.0))})
        for _ in range(int(rng.integers(1, 4))):       # several lines per key: the first one wins
            r = rng.random()
            if r < 0.2:
                mixed_scores.append(f"{key} rejected\n")
            else:
                kw = "嗨小问" if r < 0.6 else "heysnips"
                c = (round(float(rng.integers(0, 11)) / 10, 1) if rng.random() < 0.4 else float(rng.random()))
                mixed_scores.append(f"{key} detected {kw} {c:.3f}\n")
    det.append(("det_mixed", "".join(json.dumps(o, ensure_ascii=False) + "\n" for o in mixed_labels),
                "".join(mixed_scores), "嗨小问,heysnips", 0.001))
    out["ndet"] = np.array(len(det))
    for di, (name, dl, sc, kws, step) in enumerate(det):
        d = os.path.join(tmp, name)
        os.makedirs(d)
        with open(os.path.join(d, "data.list"), "w", encoding="utf8") as f:
            f.write(dl)
        with open(os.path.join(d, "score.txt"), "w", encoding="utf8") as f:
            f.write(sc)
        sys.argv = ["compute_det_ctc.py", "--test_data", os.path.join(d, "data.list"), "--keywords", escaped(kws),
                    "--score_file", os.path.join(d, "score.txt"), "--step", str(step)]
        runpy.run_path(os.path.join(REF, "wekws", "bin", "compute_det_ctc.py"), run_name="__main__")
        stats = sorted(f for f in os.listdir(d) if f.startswith("stats."))
        p = f"d{di}_"
        out.update({p + "name": np.array(name), p + "data_list": np.array(dl), p + "score": np.array(sc),
                    p + "keywords": np.array(kws), p + "step": np.array(step),
                    p + "stats_names": np.array(stats),
                    p + "stats_texts": np.array([open(os.path.join(d, f), encoding="utf8").read() for f in stats])})
        print(f"{name}: {len(stats)} stats files")
    dst = os.path.join(ROOT, "tests", "golden", "ctc_score.npz")
    save_npz(dst, out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    main()
