#!/usr/bin/env python
"""Golden vectors for the streaming CTC keyword spotter (test infrastructure): drives the REFERENCE's own
wekws/bin/stream_kws_ctc.py KeyWordSpotter (constructor, set_keywords, forward with int16 PCM bytes, reset_all) over
chunk schedules and stores what it did in tests/golden/kws_stream.npz.

    python oracle/make_kws_stream_golden.py [REFERENCE_CHECKOUT]      (default /root/reference)

The script imports two modules that are missing or unusable at the reference snapshot, so they are stubbed:
  * librosa          -- only demo() reads a wav file with it; the class never calls it;
  * tools.make_list  -- query_token_set / read_lexicon / read_token do not exist there.  read_token / read_lexicon are
                        only stored by the constructor, and set_keywords only takes (strs, indexes) from
                        query_token_set, so a stub that returns this script's token ids for each keyword gives the
                        class exactly the keywords_token / keywords_idxset it would build from real files.
The model is built by the reference's own init_model + load_checkpoint from a temporary config (the legacy
feature_extraction_conf schema the class reads) and a small GRU checkpoint, then swapped for a stub that returns
prescribed logits (CTC-like, with planted keyword token sequences) for whatever rows the front-end produced, so the
detection gates are hit on purpose.  Recorded per case: the PCM, the chunk schedule, the rows per chunk, the logits
the stub returned (the reference applies softmax(2) itself), every result dict, and a seeded sample of the feature
rows the reference computed.

Without context expansion the reference hands any wave shorter than one frame to kaldi.fbank, which asserts (window
size > samples) and drops the chunk; the schedules here avoid that case (with no context: chunks of >= 160 samples after
a first one of >= 400, so the carried 240..399 samples always complete a frame), the spotter itself returns {} for it
and carries the samples.
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"

V = 48
KEYWORDS = {"hi_xiaowen": [5, 9, 17, 23], "nihao_wenwen": [31, 7, 23, 23]}     # the second repeats a token
FILLERS = [[5, 9, 40, 17], [23, 23, 7], [31, 12]]
RESET = -1                                                                      # schedule marker: reset_all()

# name, (mel, context, skip), gates, chunk schedule spec, plant seed, sharpness
CASES = [
    # every gate: threshold, min / max duration, interval; activations in the middle of large chunks
    ("gates", dict(mel=80, context=(2, 2), skip=3), dict(threshold=0.85, min_frames=15, max_frames=33,
                                                          interval_frames=120), ("fixed", 4800, 16), 11, 9.0),
    ("compound", dict(mel=40, context=None, skip=1), dict(threshold=0.975, min_frames=5, max_frames=250,
                                                          interval_frames=30), ("fixed", 4800, 10), 12, 7.5),
    ("max_reset", dict(mel=40, context=None, skip=1), dict(threshold=0.2, min_frames=2, max_frames=25,
                                                           interval_frames=10), ("fixed", 16000, 4), 13, 8.0),
    ("left_ne_right", dict(mel=40, context=(1, 2), skip=2), dict(threshold=0.3, min_frames=4, max_frames=250,
                                                                 interval_frames=20), ("random", 1200, 6000, 14), 14, 9.0),
    ("tiny_chunks", dict(mel=40, context=None, skip=1), dict(threshold=0.3, min_frames=3, max_frames=250,
                                                             interval_frames=20), ("tiny", 40, 160), 15, 9.0),
    ("tiny_chunks_ctx", dict(mel=40, context=(2, 2), skip=3), dict(threshold=0.3, min_frames=3, max_frames=250,
                                                                   interval_frames=20), ("tiny", 50, 0), 16, 9.0),
    ("duration", dict(mel=40, context=None, skip=1), dict(threshold=0.3, min_frames=10, max_frames=16,
                                                          interval_frames=10), ("fixed", 4800, 8), 14, 9.0),
    ("reset_all", dict(mel=40, context=(2, 2), skip=3), dict(threshold=0.3, min_frames=3, max_frames=250,
                                                             interval_frames=40), ("reset", 4800, 12), 17, 9.0),
]


def stub_modules():
    sys.modules["librosa"] = types.ModuleType("librosa")
    tools = types.ModuleType("tools")
    tools.__path__ = []
    ml = types.ModuleType("tools.make_list")
    ml.read_token = lambda path: {}
    ml.read_lexicon = lambda path: {}
    # tuples, as the upstream function returns them: is_sublist compares a prefix tuple with them (:111), and a list
    # would never equal a tuple of the same length
    ml.query_token_set = lambda kw, tok, lex: (tuple(f"t{i}" for i in KEYWORDS[kw]), tuple(KEYWORDS[kw]))
    tools.make_list = ml
    sys.modules["tools"], sys.modules["tools.make_list"] = tools, ml


def schedule(spec, rng):
    kind = spec[0]
    if kind == "fixed":
        return [spec[1]] * spec[2]
    if kind == "random":
        return [int(rng.integers(spec[1], spec[2])) for _ in range(spec[3])]
    if kind == "tiny":              # chunks smaller than a frame (400 samples), empty chunks, now and then a big one
        lo = spec[2]
        out = [] if lo == 0 else [int(rng.integers(400, 1200))]
        for _ in range(spec[1]):
            r = rng.random()
            out.append(lo if r < 0.1 else int(rng.integers(max(lo, 1), 400)) if r < 0.85 else int(rng.integers(400, 3000)))
        return out
    if kind == "reset":
        n = spec[2] // 2
        return [spec[1]] * n + [RESET] + [spec[1] - 160 * 7] * n
    raise ValueError(kind)


def plant_logits(rows, seed, sharp):
    """(rows, V) logits: blank-dominated frames with keyword / filler token sequences planted, each token held 1-4 rows,
    blank gaps, an occasional competitor above the 0.05 gate."""
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(rows, V, generator=g) * 0.3
    dom = torch.zeros(rows, dtype=torch.long)
    seqs = list(KEYWORDS.values()) + FILLERS
    t = int(torch.randint(2, 10, (1,), generator=g))
    while t < rows:
        seq = seqs[int(torch.randint(0, len(seqs), (1,), generator=g))]
        hold_max = int(torch.randint(2, 6, (1,), generator=g))
        for tok in seq:
            for _ in range(int(torch.randint(1, hold_max, (1,), generator=g))):
                if t < rows:
                    dom[t] = tok
                    t += 1
            t += int(torch.randint(0, 3, (1,), generator=g))
        t += int(torch.randint(3, 25, (1,), generator=g))
    for r in range(rows):
        logits[r, dom[r]] += sharp
        if torch.rand(1, generator=g) < 0.2:
            logits[r, int(torch.randint(0, V, (1,), generator=g))] += sharp - 2.5
    return logits


def save_npz(path, arrays):
    """np.savez_compressed with fixed member timestamps, so that a rerun writes the same bytes."""
    import io
    import zipfile
    with zipfile.ZipFile(path, "w", compression=zipfile.ZIP_DEFLATED) as zf:
        for key, val in arrays.items():
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(val), allow_pickle=False)
            info = zipfile.ZipInfo(key + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            zf.writestr(info, buf.getvalue())


def main():
    stub_modules()
    sys.path.insert(0, REF)
    from wekws.bin import stream_kws_ctc as S          # noqa: E402  the reference's own module

    class StubModel(torch.nn.Module):
        """Returns the next rows of the planted logits for whatever feature rows it is given; records the features."""

        def __init__(self, logits):
            super().__init__()
            self.logits, self.pos, self.feats = logits, 0, []

        def forward(self, feature, cache):
            T = feature.size(1)
            self.feats.append(feature[0].clone())
            out = self.logits[self.pos:self.pos + T].unsqueeze(0)
            self.pos += T
            return out, cache

    out = {"V": np.array(V), "ncases": np.array(len(CASES)),
           "kw_names": np.array(list(KEYWORDS.keys())),
           "kw_tokens": np.array([t for s in KEYWORDS.values() for t in s], dtype=np.int32),
           "kw_offsets": np.cumsum([0] + [len(s) for s in KEYWORDS.values()]).astype(np.int32)}
    tmp = tempfile.mkdtemp()
    for ci, (name, fe, gates, spec, seed, sharp) in enumerate(CASES):
        rng = np.random.default_rng(seed)
        sched = schedule(spec, rng)
        total = sum(n for n in sched if n > 0)
        tt = np.arange(total)
        pcm = (1500 * np.sin(2 * np.pi * tt * (180 + 40 * ci) / 16000) + rng.normal(0, 60, total)).astype(np.int16)
        ctx = fe["context"]
        W = 1 if ctx is None else ctx[0] + ctx[1] + 1
        conf = {"dataset_conf": {"feature_extraction_conf": {"num_mel_bins": fe["mel"], "frame_length": 25,
                                                             "frame_shift": 10},
                                 "frame_skip": fe["skip"], "context_expansion": ctx is not None},
                "model": {"input_dim": fe["mel"] * W, "output_dim": V, "hidden_dim": 8,
                          "preprocessing": {"type": "linear"}, "backbone": {"type": "gru", "num_layers": 1}}}
        if ctx is not None:
            conf["dataset_conf"]["context_expansion_conf"] = {"left": ctx[0], "right": ctx[1]}
        cfg_path, ckpt = os.path.join(tmp, f"{name}.yaml"), os.path.join(tmp, f"{name}.pt")
        with open(cfg_path, "w") as f:
            yaml.safe_dump(conf, f)
        from wekws.model.kws_model import init_model
        torch.save(init_model(conf["model"]).state_dict(), ckpt)
        kws = S.KeyWordSpotter(ckpt, cfg_path, "tokens.txt", "lexicon.txt", gates["threshold"], gates["min_frames"],
                               gates["max_frames"], gates["interval_frames"], 3, 20, -1, False)
        kws.set_keywords(",".join(KEYWORDS.keys()))
        logits = plant_logits(4000, seed, sharp)
        kws.model = StubModel(logits)
        rows, res, pos = [], [], 0
        for n in sched:
            if n == RESET:
                kws.reset_all()
                rows.append(-1)
                res.append((-2, -1, np.nan, np.nan, np.nan))
                continue
            before = kws.model.pos
            r = kws.forward(pcm[pos:pos + n].astype("<i2").tobytes())
            pos += n
            rows.append(kws.model.pos - before)
            if r == {}:
                res.append((-1, -1, np.nan, np.nan, np.nan))
            elif r["state"] == 0:
                assert r["keyword"] is None and r["start"] is None and r["end"] is None and r["score"] is None
                res.append((0, -1, np.nan, np.nan, np.nan))
            else:
                res.append((1, list(KEYWORDS).index(r["keyword"]), r["start"], r["end"], r["score"]))
        used = kws.model.pos
        feats = torch.cat(kws.model.feats) if kws.model.feats else torch.zeros(0, fe["mel"] * W)
        pick = np.sort(np.random.default_rng(100 + ci).choice(len(feats), size=min(24, len(feats)), replace=False))
        res = np.array(res, dtype=np.float64)
        p = f"c{ci}_"
        out.update({p + "name": np.array(name), p + "mel": np.array(fe["mel"]),
                    p + "context": np.array(ctx if ctx is not None else (-1, -1), dtype=np.int32),
                    p + "skip": np.array(fe["skip"]),
                    p + "gates": np.array([gates["threshold"], gates["min_frames"], gates["max_frames"],
                                           gates["interval_frames"]], dtype=np.float64),
                    p + "schedule": np.array(sched, dtype=np.int32), p + "pcm": pcm,
                    p + "rows": np.array(rows, dtype=np.int32), p + "logits": logits[:used].numpy(),
                    p + "state": res[:, 0].astype(np.int32), p + "keyword": res[:, 1].astype(np.int32),
                    p + "start": res[:, 2], p + "end": res[:, 3], p + "score": res[:, 4],
                    p + "feat_idx": pick.astype(np.int32), p + "feat_rows": feats[pick].numpy()})
        print(f"{name}: {len(sched)} chunks, rows {sum(r for r in rows if r > 0)}, activations "
              f"{int((res[:, 0] == 1).sum())}, empty {int((res[:, 0] == -1).sum())}")
    dst = os.path.join(ROOT, "tests", "golden", "kws_stream.npz")
    save_npz(dst, out)
    print("wrote", dst, os.path.getsize(dst), "bytes")


if __name__ == "__main__":
    main()
