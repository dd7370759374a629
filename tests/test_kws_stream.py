"""Streaming CTC keyword spotter (wekws_b200.KeyWordSpotter, csrc/kws_stream.cu) against the reference's
stream_kws_ctc.py KeyWordSpotter: the CPU oracle (oracle/kws_stream_oracle.py) is pinned to what the reference class
returned (tests/golden/kws_stream.npz); the device spotter is checked against the oracle, results bit for bit."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import kws_oracle as O
from oracle import kws_stream_oracle as KO
from tests.conftest import golden

V_PLANT = 48
KEYWORDS = {"hi_xiaowen": {"token_id": [5, 9, 17, 23]}, "nihao_wenwen": {"token_id": [31, 7, 23, 23]}}


def _cases():
    g = golden("kws_stream")
    names = [str(n) for n in g["kw_names"]]
    kw = {n: {"token_id": g["kw_tokens"][g["kw_offsets"][i]:g["kw_offsets"][i + 1]].tolist()}
          for i, n in enumerate(names)}
    out = []
    for ci in range(int(g["ncases"])):
        p = f"c{ci}_"
        ctx = tuple(int(v) for v in g[p + "context"])
        th, mn, mx, iv = g[p + "gates"].tolist()
        results = []
        for st, k, s, e, sc in zip(g[p + "state"], g[p + "keyword"], g[p + "start"], g[p + "end"], g[p + "score"]):
            if st == -2:
                results.append(None)                                   # reset_all() marker
            elif st == -1:
                results.append({})
            elif st == 0:
                results.append({"state": 0, "keyword": None, "start": None, "end": None, "score": None})
            else:
                results.append({"state": 1, "keyword": names[int(k)], "start": float(s), "end": float(e),
                                "score": float(sc)})
        out.append(dict(name=str(g[p + "name"]), mel=int(g[p + "mel"]), context=None if ctx[0] < 0 else ctx,
                        skip=int(g[p + "skip"]), threshold=th, min_frames=int(mn), max_frames=int(mx),
                        interval_frames=int(iv), schedule=g[p + "schedule"].tolist(), pcm=g[p + "pcm"],
                        rows=g[p + "rows"].tolist(), logits=torch.from_numpy(g[p + "logits"]), results=results,
                        feat_idx=g[p + "feat_idx"], feat_rows=torch.from_numpy(g[p + "feat_rows"]), keywords=kw))
    return out


def _oracle(case, model_fn=None, fbank_fn=None):
    return KO.KeyWordSpotter(case["keywords"], case["threshold"], model_fn, num_mel_bins=case["mel"],
                             context=case["context"], frame_skip=case["skip"], min_frames=case["min_frames"],
                             max_frames=case["max_frames"], interval_frames=case["interval_frames"], fbank_fn=fbank_fn)


def _replay(case, spotter_forward, reset_all):
    """Drives one golden case's schedule; yields (chunk index, result)."""
    q = 0
    for i, n in enumerate(case["schedule"]):
        if n == -1:
            reset_all()
            continue
        yield i, spotter_forward(case["pcm"][q:q + n])
        q += n


# ----------------------------------------------------------------------------------------------------------- CPU
def test_oracle_matches_reference_golden():
    """The oracle reproduces the reference class: every result dict (score compared with ==) and the rows per chunk;
    the feature rows within the log-mel tolerance (the oracle's fbank is a restatement of torchaudio's)."""
    for case in _cases():
        pos, feats = [0], []

        def model_fn(f, cache):
            T = f.size(1)
            feats.append(f[0])
            out = case["logits"][pos[0]:pos[0] + T].unsqueeze(0)
            pos[0] += T
            return out, cache

        k = _oracle(case, model_fn)
        for i, r in _replay(case, k.forward, k.reset_all):
            assert r == case["results"][i], (case["name"], i)
        assert pos[0] == case["logits"].size(0), case["name"]
        allf = torch.cat(feats) if feats else torch.zeros(0)
        if len(case["feat_idx"]):
            err = float((allf[torch.from_numpy(case["feat_idx"]).long()] - case["feat_rows"]).abs().max())
            assert err <= 1e-3, (case["name"], err)
    # rows per chunk: the model saw exactly the golden's rows
    for case in _cases():
        got = []

        def model_fn(f, cache, case=case):
            got.append(f.size(1))
            return case["logits"][sum(got[:-1]):sum(got)].unsqueeze(0), cache

        k = _oracle(case, model_fn)
        expect = []
        for i, r in _replay(case, k.forward, k.reset_all):
            expect.append(case["rows"][i])
        assert [r for r in expect if r > 0] == got, case["name"]


def test_golden_covers_the_gates():
    cases = {c["name"]: c for c in _cases()}
    acts = sum(1 for c in cases.values() for r in c["results"] if r and r["state"] == 1)
    assert acts >= 8
    assert any(r == {} for r in cases["tiny_chunks_ctx"]["results"])
    assert 0 in cases["tiny_chunks_ctx"]["schedule"] and -1 in cases["reset_all"]["schedule"]


@pytest.mark.parametrize("context,skip", [(None, 1), ((2, 2), 3), ((1, 2), 2), ((0, 1), 1), (None, 3)])
def test_host_planning_matches_oracle_rows(context, skip):
    """StreamPlanner (the host half of the device front-end) == the oracle's accept_wave row counts, random chunks."""
    from wekws_b200.spotter import StreamPlanner
    rng = np.random.default_rng(5 + skip)
    B = 6
    pl = StreamPlanner(B, context=context, frame_skip=skip)
    oracles = [KO.KeyWordSpotter(KEYWORDS, 0.5, context=context, frame_skip=skip, num_mel_bins=23,
                                 fbank_fn=lambda w: torch.zeros(O.num_frames(w.numel()), 23)) for _ in range(B)]
    for step in range(60):
        n = rng.integers(0, 5000, B)
        if step % 17 == 5:
            pl.reset_all([2])
            oracles[2].reset_all()
        try:
            p = pl.plan(n)
        except ValueError:                  # the planner refuses the call up front; some stream's oracle asserts
            assert any(_raises(oracles[b], n[b]) for b in range(B))
            continue
        pl.commit(p)
        for b in range(B):
            f = oracles[b].accept_wave(np.zeros(n[b], np.int16))
            assert (0 if f is None else f.size(0)) == p["rows"][b], (step, b)
            assert len(oracles[b].wave_remained) == pl.carry_len[b]


def _raises(k, n):
    import copy
    try:
        copy.deepcopy(k).accept_wave(np.zeros(n, np.int16))
    except ValueError:
        return True
    return False


def test_left_greater_than_right_is_rejected():
    from wekws_b200.spotter import StreamPlanner
    with pytest.raises(ValueError):
        StreamPlanner(1, context=(2, 1))


# ----------------------------------------------------------------------------------------------------------- GPU
def _detect(state, probs_list, keywords, gates, skip, score_beam=3, path_beam=20, perm=None):
    """One wekws_kws_detect call: probs_list[b] (rows_b, V) CPU tensors; perm = order of the streams in the packed
    buffer.  Returns the (B, 6) result as a numpy array."""
    from wekws_b200 import _native
    dev = state.device
    B = len(probs_list)
    order = list(range(B)) if perm is None else list(perm)
    rows = [p.size(0) for p in probs_list]
    off, cur = [0] * B, 0
    for b in order:
        off[b] = cur
        cur += rows[b]
    V = probs_list[0].size(1)
    packed = torch.cat([probs_list[b] for b in order] + [torch.zeros(1, V)]).to(dev)
    words = list(keywords)
    seqs = [keywords[w]["token_id"] for w in words]
    toks = torch.tensor(sorted({0} | {t for s in seqs for t in s}), dtype=torch.int32, device=dev)
    kwt = torch.tensor([t for s in seqs for t in s], dtype=torch.int32, device=dev)
    kwo = torch.tensor(np.cumsum([0] + [len(s) for s in seqs]), dtype=torch.int32, device=dev)
    d_off = torch.tensor(off, dtype=torch.int32, device=dev)
    d_rows = torch.tensor(rows, dtype=torch.int32, device=dev)
    res = torch.empty(B, 6, dtype=torch.int64, device=dev)
    cfg = _native.KwsConfig(float(gates["threshold"]), gates["min_frames"], gates["max_frames"],
                            gates["interval_frames"], score_beam, path_beam, skip)

    def p(t):
        return C.c_void_p(t.data_ptr())

    _native.check(_native.lib().wekws_kws_detect(p(packed), p(d_off), p(d_rows), B, V, p(toks), toks.numel(), p(kwt),
                                                 p(kwo), len(words), C.byref(cfg), p(state), p(res),
                                                 C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                  "wekws_kws_detect")
    return res.cpu().numpy()


def _kws_state(B, dev="cuda"):
    from wekws_b200 import _native
    st = torch.zeros(B, int(_native.lib().wekws_kws_state_bytes()), dtype=torch.uint8, device=dev)
    _reset(st, None, True)
    return st


def _reset(st, ids, full):
    from wekws_b200 import _native
    d = None if ids is None else torch.tensor(ids, dtype=torch.int32, device=st.device)
    _native.check(_native.lib().wekws_kws_reset(C.c_void_p(st.data_ptr()), st.size(0),
                                                None if d is None else C.c_void_p(d.data_ptr()),
                                                0 if d is None else len(ids), 1 if full else 0,
                                                C.c_void_p(torch.cuda.current_stream().cuda_stream)), "wekws_kws_reset")


def _as_dict(r, words, resolution=0.01):
    if r[0] < 0:
        return {}
    if r[0] == 0:
        return {"state": 0, "keyword": None, "start": None, "end": None, "score": None}
    return {"state": 1, "keyword": words[int(r[1])], "start": int(r[2]) * resolution, "end": int(r[3]) * resolution,
            "score": float(np.array([r[4]], dtype=np.int64).view(np.float64)[0])}


@pytest.mark.gpu
def test_device_detect_on_golden_probs():
    """wekws_kws_detect fed the probabilities the reference computed reproduces every result of every golden case."""
    for case in _cases():
        st = _kws_state(1)
        probs = case["logits"].unsqueeze(0).softmax(2)[0]
        pos = 0
        words = list(case["keywords"])
        gates = {k: case[k] for k in ("threshold", "min_frames", "max_frames", "interval_frames")}
        for i, n in enumerate(case["schedule"]):
            if n == -1:
                _reset(st, None, True)
                continue
            r = case["rows"][i]
            res = _detect(st, [probs[pos:pos + r]], case["keywords"], gates, case["skip"])
            pos += r
            assert _as_dict(res[0], words) == case["results"][i], (case["name"], i)
            assert res[0][5] == 0


def _plant(rows, seed, sharp=9.0):
    from oracle.make_kws_stream_golden import plant_logits
    return plant_logits(rows, seed, sharp).unsqueeze(0).softmax(2)[0]


def _run_streams(B, seed, calls, gates, skip, resets=(), batch_split=1):
    """B streams of planted posteriors in ragged chunks (0..24 rows), packed in a random stream order, against one
    oracle per stream.  resets: {call index: (ids, full)}."""
    rng = np.random.default_rng(seed)
    probs = [_plant(24 * calls, 1000 + b) for b in range(B)]
    pos = [0] * B
    orc = [KO.KeyWordSpotter(KEYWORDS, gates["threshold"], frame_skip=skip, min_frames=gates["min_frames"],
                             max_frames=gates["max_frames"], interval_frames=gates["interval_frames"])
           for _ in range(B)]
    st = _kws_state(B)
    words = list(KEYWORDS)
    activations = 0
    for c in range(calls):
        if c in resets:
            ids, full = resets[c]
            _reset(st, ids, full)
            for b in ids:
                (orc[b].reset_all if full else orc[b].reset)()
        rows = rng.integers(0, 25, B)
        chunks = [probs[b][pos[b]:pos[b] + rows[b]] for b in range(B)]
        for b in range(B):
            pos[b] += int(rows[b])
        if batch_split == 1:
            res = _detect(st, chunks, KEYWORDS, gates, skip, perm=rng.permutation(B))
        else:
            n = B // batch_split
            res = np.concatenate([_detect(st[i * n:(i + 1) * n], chunks[i * n:(i + 1) * n], KEYWORDS, gates, skip)
                                  for i in range(batch_split)])
        for b in range(B):
            want = orc[b].forward_probs(chunks[b])
            assert _as_dict(res[b], words) == want, (c, b)
            activations += want.get("state", 0)
    return activations


GATES = dict(threshold=0.3, min_frames=3, max_frames=80, interval_frames=20)


@pytest.mark.gpu
def test_device_detect_many_streams_ragged_permuted():
    assert _run_streams(257, 3, 8, GATES, skip=3) > 20


@pytest.mark.gpu
def test_device_reset_and_reset_all_part_way():
    B = 64
    resets = {3: (list(range(0, B, 3)), False), 5: (list(range(1, B, 4)), True), 6: (list(range(B)), False)}
    assert _run_streams(B, 4, 9, GATES, skip=1, resets=resets) > 0


@pytest.mark.gpu
def test_device_detect_4096_streams_equals_four_calls_of_1024():
    torch.manual_seed(0)
    B = 4096
    probs = [_plant(30, 7000 + b % 97) for b in range(B)]
    a = _detect(_kws_state(B), probs, KEYWORDS, GATES, 1)
    st = _kws_state(B)
    b4 = np.concatenate([_detect(st[i * 1024:(i + 1) * 1024], probs[i * 1024:(i + 1) * 1024], KEYWORDS, GATES, 1)
                         for i in range(4)])
    assert np.array_equal(a, b4) and (a[:, 0] == 1).sum() > 0


@pytest.mark.gpu
def test_prefix_overflow_is_reported():
    """A stream whose prefix outgrows WEKWS_CTC_MAX_PREFIX tokens is flagged; the others are not."""
    T = 80
    good = _plant(T, 1)
    bad = torch.full((T, V_PLANT), 1e-4)
    for t in range(T):
        bad[t, 5 if t % 2 == 0 else 9] = 1.0                              # 5 9 5 9 ...: the prefix grows every frame
    bad = bad / bad.sum(1, keepdim=True)
    gates = dict(GATES, max_frames=10_000)
    res = _detect(_kws_state(2), [good, bad], KEYWORDS, gates, 1)
    assert res[0][5] == 0 and res[1][5] == 1


KW_TOKENS = (0, 5, 7, 9, 17, 23, 31)


def _peaky_model(name, seed, feats):
    """Random fsmn (shipped size: 80 x (2+1+2) inputs, odim 2599) or ds_tcn (40 mel, identity, odim 2599) whose output
    layer only scores blank and the keyword tokens, scaled on `feats` so that those logits spread by ~6: the posteriors
    are peaky enough for the beam to move (random weights over 2599 outputs never get a token above 0.05)."""
    from wekws_b200 import init_model, model_config, synth
    if name == "fsmn":
        cfg = model_config("fsmn", input_dim=400, output_dim=2599)
    else:
        cfg = model_config("ds_tcn", input_dim=40, output_dim=2599, activation="identity")
    model = synth.randomize_(init_model(cfg), seed=seed).eval()
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        last = [m for m in model.modules() if isinstance(m, torch.nn.Linear)][-1]
        last.weight.zero_()
        last.bias.zero_()
        for t in KW_TOKENS:
            last.weight[t] = torch.randn(last.weight.size(1), generator=g)
        sd = {k: v.clone() for k, v in model.state_dict().items()}
        y, _ = O.kws_forward(sd, cfg, feats, None)
        last.weight.mul_(6.0 / float(y[..., list(KW_TOKENS)].std()))
        last.bias[list(KW_TOKENS)] = 8.0
    return cfg, model


def _features_oracle(sd, cfg, **kw):
    """Oracle spotter whose model is the oracle model (kws_forward); probabilities recorded."""
    seen = []

    def model_fn(f, cache):
        y, c = O.kws_forward(sd, cfg, f, cache)
        seen.append(y.softmax(2)[0])
        return y, c
    return model_fn, seen


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fsmn", "ds_tcn"])
def test_end_to_end_pcm_to_results(name):
    """PCM -> results.  Device features == the oracle's accept_wave on the device Fbank rows bit for bit (rows and
    counts exact) and within the log-mel tolerance of the oracle's own fbank; posteriors within 1e-4 of the oracle
    model on the oracle's features; results == the oracle decoder on the device's own posteriors, bit for bit."""
    from wekws_b200 import Fbank, KeyWordSpotter, synth
    mel, context, skip = (80, (2, 2), 3) if name == "fsmn" else (40, None, 1)
    B = 5
    pcm = synth.pcm_int16(B, 16000 * 4, seed=9)
    f0 = O.fbank(pcm[0, :16000].float(), num_mel_bins=mel)
    if context is not None:
        f0 = O.context_expansion(f0, *context)
    cfg, model = _peaky_model(name, 11, f0.unsqueeze(0))
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.cuda()
    kws = dict(min_frames=2, max_frames=100, interval_frames=20)
    sp = KeyWordSpotter(model, KEYWORDS, 0.05, B, "cuda", num_mel_bins=mel, context=context, frame_skip=skip, **kws)
    fb = Fbank(mel)
    dev_fbank = lambda w: fb(w.to(torch.int16).cuda()).cpu()                       # noqa: E731
    ora_dev = [KO.KeyWordSpotter(KEYWORDS, 0.05, num_mel_bins=mel, context=context, frame_skip=skip,
                                 fbank_fn=dev_fbank, **kws) for _ in range(B)]
    ora_ref = [KO.KeyWordSpotter(KEYWORDS, 0.05, num_mel_bins=mel, context=context, frame_skip=skip, **kws)
               for _ in range(B)]
    dec = [KO.KeyWordSpotter(KEYWORDS, 0.05, frame_skip=skip, **kws) for _ in range(B)]
    caches = [None] * B
    rng = np.random.default_rng(2)
    q = [0] * B
    advanced = False
    for c in range(14):
        n = rng.integers(900, 6000, B) if c % 3 else np.full(B, 4800)
        N = int(n.max())
        chunk = torch.zeros(B, N, dtype=torch.int16)
        for b in range(B):
            chunk[b, :n[b]] = pcm[b, q[b]:q[b] + n[b]]
            q[b] += int(n[b])
        res = sp.forward(chunk.cuda(), lengths=n.tolist())
        feats, probs = sp.features.cpu(), sp.probs.cpu()
        for b in range(B):
            f_dev = ora_dev[b].accept_wave(chunk[b, :n[b]].numpy())
            f_ref = ora_ref[b].accept_wave(chunk[b, :n[b]].numpy())
            r0, nr = int(sp.row_offsets[b]), int(sp.rows[b])
            rows_o = 0 if f_dev is None else f_dev.size(0)
            assert nr == rows_o and (f_ref is None) == (f_dev is None)
            if nr == 0:
                assert res[b] == {}
                continue
            assert torch.equal(feats[r0:r0 + nr], f_dev), (c, b)
            assert float((f_ref - f_dev).abs().max()) <= 1e-3, (c, b)
            y_ref, caches[b] = O.kws_forward(sd, cfg, f_dev.unsqueeze(0), caches[b])
            assert float((probs[r0:r0 + nr] - y_ref.softmax(2)[0]).abs().max()) <= 1e-4, (c, b)
            want = dec[b].forward_probs(probs[r0:r0 + nr])
            assert res[b] == want, (c, b)
            advanced |= any(len(h[0]) > 0 for h in dec[b].cur_hyps) or want.get("state", 0) == 1
    assert advanced, "the planted-peaky model never moved the beam"


@pytest.mark.gpu
def test_spliced_chunked_fbank_equals_whole_wave_fbank():
    """No context, no skip: the rows of all chunks back to back == one Fbank call over the whole waveform."""
    from wekws_b200 import Fbank, KeyWordSpotter, init_model, model_config, synth
    model = synth.randomize_(init_model(model_config("ds_tcn", input_dim=40, output_dim=20, activation="identity")))
    sp = KeyWordSpotter(model.eval().cuda(), KEYWORDS, 0.5, 2, "cuda", num_mel_bins=40)
    pcm = synth.pcm_int16(2, 20000, seed=4)
    rng = np.random.default_rng(1)
    rows = [[], []]
    q = 0
    while q < 20000:
        n = int(min(rng.integers(100, 3000), 20000 - q))
        sp.forward(pcm[:, q:q + n].cuda())
        q += n
        for b in range(2):
            r0, nr = int(sp.row_offsets[b]), int(sp.rows[b])
            rows[b].append(sp.features[r0:r0 + nr].cpu())
    whole = Fbank(40)(pcm.cuda()).cpu()
    for b in range(2):
        got = torch.cat(rows[b])
        assert got.size(0) == whole.size(1) and torch.equal(got, whole[b])


@pytest.mark.gpu
def test_forward_async_makes_no_host_sync_and_launch_count():
    from wekws_b200 import KeyWordSpotter, _native, init_model, model_config, synth
    model = synth.randomize_(init_model(model_config("fsmn", input_dim=400, output_dim=64))).eval().cuda()
    B = 8
    sp = KeyWordSpotter(model, KEYWORDS, 0.5, B, "cuda", context=(2, 2), frame_skip=3)
    pcm = synth.pcm_int16(B, 4800, seed=3).cuda()
    sp.forward(pcm)                                                     # warm-up (packs the model, Fbank tables)
    n0 = _native.launch_count()
    model.forward_softmax(torch.zeros(3, 9, 400, device="cuda"))
    torch.cuda.synchronize()
    per_model = _native.launch_count() - n0
    sp.reset_all([1, 2])                                                 # streams 1, 2 restart: ragged row counts
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        n0 = _native.launch_count()
        out = sp.forward_async(pcm, lengths=[2400] + [4800] * (B - 1))
        launches = _native.launch_count() - n0
    finally:
        torch.cuda.set_sync_debug_mode(0)
    groups = len(set(int(r) for r in sp.rows if r > 0))
    assert groups >= 2
    assert launches <= 4 + groups * per_model
    assert out.shape == (B, 6)
