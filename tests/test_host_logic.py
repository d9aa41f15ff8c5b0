"""CPU: host-side logic of the product package (no GPU, no kernels): option handling, initial tokens,
suppress lists, hypothesis finalisation / ranking, window splitting, padding, id tables."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from helpers import GOLD


def fake_model(name):
    from whisper_b200 import synthetic
    from whisper_b200.model import ModelDimensions

    dims = ModelDimensions(**synthetic.dims_dict(name))
    return SimpleNamespace(dims=dims, is_multilingual=dims.n_vocab >= 51865,
                           num_languages=dims.n_vocab - 51765 - int(dims.n_vocab >= 51865),
                           device=torch.device("cpu"), dtype=torch.float16)


def test_mel_filterbank_regenerated_bit_exact():
    from whisper_b200.audio import _slaney_mel_filterbank

    g = np.load(os.path.join(GOLD, "mel_filters.npz"))
    for n in (80, 128):
        assert np.array_equal(_slaney_mel_filterbank(n), g[f"mel_{n}"])


def test_tokenizer_ids_match_reference_table():
    from whisper_b200.tokenizer import get_tokenizer

    with open(os.path.join(GOLD, "token_ids.json")) as f:
        table = json.load(f)
    for n_vocab, spec in table["specials"].items():
        n_vocab = int(n_vocab)
        multi = n_vocab >= 51865
        tk = get_tokenizer(multi, num_languages=n_vocab - 51765 - int(multi), language="en", task="transcribe")
        for k in ("eot", "sot", "translate", "transcribe", "sot_lm", "sot_prev", "no_speech", "no_timestamps",
                  "timestamp_begin"):
            assert getattr(tk, k) == spec[k], (n_vocab, k)
        assert list(tk.sot_sequence) == spec["sot_sequence"]
        assert tk.n_vocab == n_vocab
        assert sorted(tk.all_language_tokens) == sorted(spec["all_language_tokens"])
        assert len(tk.non_speech_tokens) == spec["n_non_speech"]


@pytest.mark.parametrize("name", ["test-en", "test-multi"])
@pytest.mark.parametrize("opts", [
    dict(), dict(without_timestamps=True), dict(prompt=list(range(1000, 1300))), dict(prefix=[5, 6, 7], sample_len=100),
    dict(suppress_tokens="", suppress_blank=False), dict(suppress_tokens="-1,17,23"), dict(beam_size=5, patience=2.0),
    dict(max_initial_timestamp=None), dict(prompt=[1, 2, 3], prefix=[9, 9]),
])
def test_task_setup_matches_oracle(name, opts):
    from oracle import decoding as OD
    from whisper_b200.decoding import DecodingOptions, DecodingTask

    model = fake_model(name)
    task = DecodingTask(model, DecodingOptions(language="en", **opts))
    o = dict(opts)
    st = o.get("suppress_tokens", "-1")
    if isinstance(st, str):
        o["suppress_tokens"] = tuple(int(t) for t in st.split(",")) if st else ()
    oopt = OD.Options(**o)
    ids = OD.token_ids(model.dims.n_vocab)
    sample_len = oopt.sample_len or model.dims.n_text_ctx // 2
    assert task.initial_tokens == OD.initial_tokens(ids, oopt, model.dims.n_text_ctx, sample_len)
    assert tuple(task.suppress) == (OD.suppress_list(ids, oopt) if oopt.suppress_tokens else ())
    cfg = task.session_config(3)
    assert cfg["n_init"] == len(task.initial_tokens) and cfg["sot_index"] == task.initial_tokens.index(ids.sot)
    assert cfg["timestamp_rules"] == int(not oopt.without_timestamps)
    if oopt.beam_size:
        assert cfg["max_candidates"] == round(oopt.beam_size * (oopt.patience or 1.0)) and cfg["n_group"] == oopt.beam_size
    exp_mits = -1
    if not oopt.without_timestamps and oopt.max_initial_timestamp:
        exp_mits = round(oopt.max_initial_timestamp / 0.02)
    assert cfg["max_initial_timestamp_index"] == exp_mits


def test_option_validation_errors():
    from whisper_b200.decoding import DecodingOptions, DecodingTask

    m = fake_model("test-en")
    for bad in (dict(beam_size=5, best_of=5), dict(best_of=3), dict(patience=1.0), dict(length_penalty=1.5)):
        with pytest.raises(ValueError):                        # decoding.py:572-585
            DecodingTask(m, DecodingOptions(language="en", **bad))
    # temperature together with beam_size: the reference builds a BeamSearchDecoder and only records the temperature
    # (decoding.py:548-552), so decode(..., beam_size=5, temperature=0.2) must be accepted
    both = DecodingTask(m, DecodingOptions(language="en", temperature=0.4, beam_size=5)).session_config(2)
    assert both["beam_search"] == 1 and both["n_group"] == 5
    with pytest.raises(ValueError):
        DecodingTask(m, DecodingOptions(language="en", temperature=-0.1))
    task = DecodingTask(m, DecodingOptions(language="en", temperature=0.4, best_of=3))
    cfg = task.session_config(2)
    assert cfg["n_group"] == 3 and cfg["beam_search"] == 0     # decoding.py:524-526


def test_finalize_and_rank_match_oracle():
    from oracle import decoding as OD
    from whisper_b200.decoding import DecodingOptions, DecodingTask

    m = fake_model("test-en")
    rng = np.random.RandomState(3)
    for alpha in (None, 0.6):
        task = DecodingTask(m, DecodingOptions(language="en", beam_size=4, length_penalty=alpha))
        ids = OD.token_ids(m.dims.n_vocab)
        B, G, L, ctx, mc = 3, 4, 9, m.dims.n_text_ctx, 4
        tokens = rng.randint(0, 50000, size=(B, G, L))
        lp = rng.randn(B, G).astype(np.float32)
        fin_count = np.array([0, 2, 4])
        fin_tokens = np.zeros((B, mc, ctx), dtype=np.int32)
        fin_len = np.zeros((B, mc), dtype=np.int32)
        fin_score = rng.randn(B, mc).astype(np.float32)
        beam = OD.BeamState(G, ids.eot, None)
        beam.finished = [dict() for _ in range(B)]
        for a in range(B):
            for k in range(fin_count[a]):
                n = 4 + k
                seq = rng.randint(0, 50000, size=n).tolist() + [ids.eot]
                fin_tokens[a, k, : n + 1] = seq
                fin_len[a, k] = n + 1
                beam.finished[a][tuple(seq)] = float(fin_score[a, k])
        cands, scores = task._finalize(tokens, lp, (fin_tokens, fin_len, fin_score, fin_count))
        o_c, o_s = beam.finalize([[tokens[a, j].tolist() for j in range(G)] for a in range(B)], torch.from_numpy(lp))
        assert cands == o_c and scores == o_s
        sb = 1
        sliced = [[s[sb: s.index(ids.eot)] for s in grp] for grp in cands]
        assert task._rank(sliced, scores) == OD.rank(sliced, scores, alpha)


def test_pad_or_trim():
    from oracle import audio as OA
    from whisper_b200.audio import pad_or_trim

    x = np.arange(10, dtype=np.float32).reshape(2, 5)
    for n in (3, 5, 8):
        assert np.array_equal(pad_or_trim(x, n), OA.pad_or_trim(x, n))
        assert np.array_equal(pad_or_trim(torch.from_numpy(x), n).numpy(), OA.pad_or_trim(x, n))
        assert np.array_equal(pad_or_trim(torch.from_numpy(x), n, axis=0).numpy(), OA.pad_or_trim(x, n, axis=0))


def test_window_splitting_rules():
    """transcribe.py:339-399 on handcrafted token rows (tb = timestamp_begin)."""
    from whisper_b200.decoding import DecodingResult
    from whisper_b200.tokenizer import get_tokenizer
    from whisper_b200.transcribe import _WindowLoop

    tk = get_tokenizer(False)
    tb = tk.timestamp_begin
    loop = _WindowLoop.__new__(_WindowLoop)
    loop.tokenizer, loop.input_stride, loop.time_precision = tk, 2, 0.02

    def res(tokens):
        return DecodingResult(audio_features=None, language="en", tokens=tokens, temperature=0.0, avg_logprob=-0.1,
                              compression_ratio=1.0, no_speech_prob=0.0)

    # two complete segments then an unfinished one: seek advances to the last consecutive pair's timestamp
    toks = [tb, 11, 12, tb + 100, tb + 100, 13, tb + 250, tb + 250, 14]
    segs, seek = loop.split_window(0, 3000, 30.0, res(toks))
    assert [s["tokens"] for s in segs] == [[tb, 11, 12, tb + 100], [tb + 100, 13, tb + 250]]
    assert (segs[0]["start"], segs[0]["end"]) == (0.0, 2.0) and segs[1]["end"] == 5.0
    assert seek == 250 * 2
    # single timestamp ending: the tail is kept and the whole window is consumed
    toks = [tb, 11, tb + 100, tb + 100, 12, tb + 400]
    segs, seek = loop.split_window(1000, 3000, 30.0, res(toks))
    assert [s["tokens"] for s in segs] == [[tb, 11, tb + 100], [tb + 100, 12, tb + 400]] and seek == 4000
    assert segs[1]["start"] == pytest.approx(10.0 + 2.0) and segs[1]["end"] == pytest.approx(10.0 + 8.0)
    # no consecutive timestamps: one segment, duration from the last timestamp
    segs, seek = loop.split_window(0, 2000, 20.0, res([tb, 11, 12, tb + 300]))
    assert len(segs) == 1 and segs[0]["end"] == pytest.approx(6.0) and seek == 2000
    segs, seek = loop.split_window(0, 2000, 20.0, res([11, 12]))
    assert segs[0]["end"] == pytest.approx(20.0)


def test_temperature_fallback_ladder():
    """transcribe.py:184-224: walk the temperature ladder until the result passes the compression-ratio /
    log-prob checks; beam options are dropped above temperature 0, best_of at 0; silence keeps a bad result."""
    from whisper_b200.decoding import DecodingResult
    from whisper_b200.transcribe import _WindowLoop

    calls = []

    class FakeModel:
        def __init__(self, script):
            self.script = script

        def decode(self, segment, options):
            calls.append(options)
            cr, lp, ns = self.script[min(len(calls) - 1, len(self.script) - 1)]
            return DecodingResult(audio_features=None, language="en", tokens=[1], temperature=options.temperature,
                                  avg_logprob=lp, compression_ratio=cr, no_speech_prob=ns)

    def make(script, **kw):
        calls.clear()
        loop = _WindowLoop.__new__(_WindowLoop)
        loop.model = FakeModel(script)
        loop.temperatures = [0.0, 0.2, 0.4]
        loop.cr_threshold, loop.lp_threshold, loop.ns_threshold = 2.4, -1.0, 0.6
        loop.decode_options = dict(language="en", beam_size=5, patience=1.0, best_of=3, **kw)
        return loop

    # first rung too repetitive, second has a low log-prob, third is fine
    r = make([(3.0, -0.2, 0.0), (1.0, -1.5, 0.0), (1.0, -0.3, 0.0)]).decode_with_fallback(None)
    assert r.temperature == 0.4 and len(calls) == 3
    assert calls[0].beam_size == 5 and calls[0].best_of is None and calls[0].temperature == 0.0
    assert calls[1].beam_size is None and calls[1].patience is None and calls[1].best_of == 3
    # a good first rung stops the ladder
    r = make([(1.0, -0.3, 0.0)]).decode_with_fallback(None)
    assert r.temperature == 0.0 and len(calls) == 1
    # low log-prob but probably silence: accepted as is (transcribe.py:216-222)
    r = make([(1.0, -1.5, 0.9), (1.0, -0.1, 0.0)]).decode_with_fallback(None)
    assert r.temperature == 0.0 and len(calls) == 1
    # nothing passes: the last rung's result is returned
    r = make([(3.0, -0.2, 0.0)]).decode_with_fallback(None)
    assert r.temperature == 0.4 and len(calls) == 3


def _fake_decode_fn(tb):
    """A deterministic stand-in for the device decode: tokens / quality numbers are a pure function of the window's
    content, the prompt and the temperature, with timestamps that move the seek position by different amounts."""
    from whisper_b200.decoding import DecodingResult

    def fake(segment, options):
        h = int(abs(float(segment.double().sum())) * 1000) % 97
        p = len(options.prompt or [])
        t_end = 100 + (h * 13 + p) % 1300
        tokens = [tb, 1000 + h, 1001 + (p % 7), tb + t_end // 2, tb + t_end // 2, 2000 + h, tb + t_end]
        if h % 3 == 0:
            tokens = tokens[:-1]                         # ends in text: seek goes to the last timestamp pair
        bad = (h % 5 == 0) and options.temperature < 0.4
        return DecodingResult(audio_features=None, language="en", tokens=tokens, temperature=options.temperature,
                              avg_logprob=-1.5 if bad else -0.2, compression_ratio=1.0, no_speech_prob=0.1)

    return fake


def test_transcribe_batch_equals_per_file_transcribe(monkeypatch):
    """transcribe_batch (SURVEY.md 8f.1) advances many files' window loops in lock-step; with a deterministic
    decoder every file must get exactly what transcribe() gives it alone, requests must be batched across files,
    and requests sharing a session must have prompts of one length."""
    from oracle import audio as OA
    import importlib

    import whisper_b200.decoding as WD
    from whisper_b200.tokenizer import get_tokenizer

    WT = importlib.import_module("whisper_b200.transcribe")     # the package attribute of that name is the function

    def cpu_mel(audio, n_mels=80, padding=0, device=None):
        return torch.from_numpy(OA.log_mel_spectrogram(np.asarray(audio, dtype=np.float32), n_mels, padding).astype(np.float32))

    monkeypatch.setattr(WT, "log_mel_spectrogram", cpu_mel)
    tb = get_tokenizer(False).timestamp_begin
    fake = _fake_decode_fn(tb)
    model = fake_model("test-en")
    model.decode = fake
    rng = np.random.RandomState(5)
    audios = [rng.randn(16000 * secs).astype(np.float32) * 0.1 for secs in (95, 31, 64, 140, 8)]
    kw = dict(temperature=(0.0, 0.4), no_speech_threshold=0.6, logprob_threshold=-1.0)
    alone = [WT.transcribe(model, a, **kw) for a in audios]
    assert sum(len(r["segments"]) for r in alone) > 12

    batches = []

    def fake_requests(m, requests, max_batch=64):
        tasks_len = {}
        for seg, opt in requests:
            tasks_len.setdefault((len(opt.prompt or []), opt.temperature), 0)
            tasks_len[(len(opt.prompt or []), opt.temperature)] += 1
        batches.append((len(requests), len(tasks_len)))
        return [fake(seg, opt) for seg, opt in requests]

    monkeypatch.setattr(WD, "decode_requests", fake_requests)
    together = WT.transcribe_batch(model, audios, **kw)
    for a, b in zip(alone, together):
        assert a["text"] == b["text"] and a["language"] == b["language"]
        assert [(s["seek"], s["start"], s["end"], s["tokens"], s["temperature"]) for s in a["segments"]] == \
               [(s["seek"], s["start"], s["end"], s["tokens"], s["temperature"]) for s in b["segments"]]
    rounds = together[0]["rounds"]
    assert rounds == len(batches) and batches[0][0] == len(audios)
    n_requests = sum(n for n, _ in batches)
    assert rounds < n_requests                            # the files really shared rounds
    assert transcribe_is_single_request_stream(WT, model, audios[1], kw, fake)


def transcribe_is_single_request_stream(WT, model, audio, kw, fake):
    """A one-file batch issues the same request sequence as transcribe()."""
    seen = []
    model.decode = lambda seg, opt: (seen.append(("single", len(opt.prompt or []), opt.temperature)), fake(seg, opt))[1]
    WT.transcribe(model, audio, **kw)
    single = [x[1:] for x in seen]
    seen.clear()
    import whisper_b200.decoding as WD
    WD_decode = WD.decode_requests
    try:
        WD.decode_requests = lambda m, reqs, max_batch=64: [
            (seen.append(("batch", len(o.prompt or []), o.temperature)), fake(s, o))[1] for s, o in reqs]
        WT.transcribe_batch(model, [audio], **kw)
    finally:
        WD.decode_requests = WD_decode
    return single == [x[1:] for x in seen]


def test_decode_requests_groups_by_prompt_length(monkeypatch):
    """decoding.decode_requests: requests with equal options and equally long prompts share one session (each row
    prefilled with its own prompt); a different prompt length, temperature or beam size opens another."""
    import whisper_b200.decoding as WD

    model = fake_model("test-en")
    runs = []

    def fake_run(self, mel, initial_tokens=None):
        runs.append((mel.shape[0], initial_tokens.copy(), self.options.temperature, self.options.beam_size))
        return [WD.DecodingResult(audio_features=None, language="en", tokens=[int(initial_tokens[i, 1])])
                for i in range(mel.shape[0])]

    monkeypatch.setattr(WD.DecodingTask, "run", fake_run)
    seg = torch.zeros(80, 3000)
    O = WD.DecodingOptions
    reqs = [(seg, O(language="en", prompt=[11, 12, 13])), (seg, O(language="en", prompt=[21, 22])),
            (seg, O(language="en", prompt=[31, 32, 33])), (seg, O(language="en", prompt=[41, 42, 43], temperature=0.2)),
            (seg, O(language="en", prompt=[51, 52, 53], beam_size=2)), (seg, O(language="en", prompt=[61, 62, 63]))]
    out = WD.decode_requests(model, reqs, max_batch=2)
    assert [r.tokens[0] for r in out] == [11, 21, 31, 41, 51, 61]          # request order kept, own prompt per row
    sizes = sorted(n for n, _, _, _ in runs)
    assert sizes == [1, 1, 1, 1, 2]                                         # {11,31} share (max_batch 2), 61 overflows
    for n, init, _, _ in runs:
        assert init.shape[0] == n and (init[:, 0] == init[0, 0]).all()      # <|startofprev|> first in every row


def _replay_transcribe_case(case, monkeypatch):
    """Drive OUR window loop with the decode results the REFERENCE's transcribe() run recorded (tests/golden/
    transcribe_*.json, made by oracle/make_golden.py: gen_transcribe).  Every request our loop issues must be the one
    the reference issued at that point - same prompt tokens, temperature, beam / best_of switching, same window of
    the spectrogram - and the final segments must be the reference's."""
    import importlib

    from oracle import audio as OA
    from whisper_b200 import synthetic
    from whisper_b200.decoding import DecodingResult
    from whisper_b200.tokenizer import get_tokenizer

    WT = importlib.import_module("whisper_b200.transcribe")
    with open(os.path.join(GOLD, "transcribe_test-multi.json")) as f:
        gold = json.load(f)
    c = gold["cases"][case]
    audio = synthetic.synthetic_audio(1, 16000 * c["seconds"], seed=c["audio_seed"], kind=c["audio_kind"])[0]

    def cpu_mel(a, n_mels=80, padding=0, device=None):
        return torch.from_numpy(OA.log_mel_spectrogram(np.asarray(a, dtype=np.float32), n_mels, padding).astype(np.float32))

    monkeypatch.setattr(WT, "log_mel_spectrogram", cpu_mel)
    model = fake_model(gold["model"])
    tok = get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en", task="transcribe")
    texts = c["texts"]
    monkeypatch.setattr(tok, "decode", lambda ids, **kw: texts[",".join(str(int(t)) for t in ids)])
    calls = iter(c["calls"])
    n_seen = [0]

    def decode(segment, options):
        want = next(calls)
        n_seen[0] += 1
        assert list(options.prompt or []) == want["prompt"], f"call {n_seen[0]}: prompt differs"
        assert options.temperature == pytest.approx(want["temperature"])
        assert (options.beam_size, options.best_of, options.patience) == (want["beam_size"], want["best_of"], want["patience"])
        assert options.sample_len == want["sample_len"]
        assert float(segment.double().abs().sum()) == pytest.approx(want["window_abs"], rel=2e-4), \
            f"call {n_seen[0]}: a different window of the spectrogram was decoded"
        return DecodingResult(audio_features=None, language="en", tokens=want["tokens"], text="",
                              avg_logprob=want["avg_logprob"], no_speech_prob=want["no_speech_prob"],
                              temperature=want["result_temperature"], compression_ratio=want["compression_ratio"])

    model.decode = decode
    kw = dict(c["kwargs"])
    if isinstance(kw.get("temperature"), list):
        kw["temperature"] = tuple(kw["temperature"])
    out = WT.transcribe(model, audio, language="en", **kw)
    assert n_seen[0] == len(c["calls"]), "our loop issued fewer decode requests than the reference"
    assert out["language"] == c["language"] and out["text"] == c["text"]
    assert len(out["segments"]) == len(c["segments"])
    for ours, ref in zip(out["segments"], c["segments"]):
        assert (ours["id"], ours["seek"], ours["tokens"], ours["text"]) == (ref["id"], ref["seek"], ref["tokens"], ref["text"])
        assert ours["start"] == pytest.approx(ref["start"], abs=1e-6) and ours["end"] == pytest.approx(ref["end"], abs=1e-6)
        for k in ("temperature", "avg_logprob", "compression_ratio", "no_speech_prob"):
            assert ours[k] == pytest.approx(ref[k])


@pytest.mark.parametrize("case", ["ladder_conditioned", "ladder_compression", "greedy_unconditioned", "beam_clips",
                                  "silence_skip", "no_thresholds"])
def test_transcribe_window_loop_replays_reference(case, monkeypatch):
    _replay_transcribe_case(case, monkeypatch)


def test_checkpoint_keys_and_weight_packing():
    """Checkpoint ingest (reference __init__.py:147-156 -> model.load_state_dict): the tensors a released checkpoint
    holds - names and shapes of the REFERENCE's Whisper.state_dict(), tests/golden/state_dict_keys.json - are exactly
    the ones whisper_b200 expects, pack_weights() consumes every one of them, and the packed slots have the layout
    include/whisper_b200.h documents (tap-major conv weights, fused q|k|v with a zero key bias, fp32 LayerNorms)."""
    from whisper_b200 import synthetic
    from whisper_b200.model import ModelDimensions, pack_weights

    with open(os.path.join(GOLD, "state_dict_keys.json")) as f:
        ref_keys = json.load(f)
    for name, shapes in ref_keys.items():
        spec = {n: list(s) for n, s, _ in synthetic.state_dict_spec(synthetic.dims_dict(name))}
        assert spec == shapes, f"{name}: state dict layout differs from the reference"

    class Tracking(dict):
        def __init__(self, *a):
            super().__init__(*a)
            self.read = set()

        def __getitem__(self, k):
            self.read.add(k)
            return super().__getitem__(k)

    for name in ("test-en", "test-multi", "tiny.en"):
        dd = synthetic.dims_dict(name)
        dims = ModelDimensions(**dd)
        sd = Tracking(synthetic.synthetic_state_dict(dd, seed=3))
        packed = pack_weights(sd, dims, "cpu", torch.float16)
        assert sd.read == set(ref_keys[name]), f"{name}: unread checkpoint tensors {set(ref_keys[name]) - sd.read}"
        assert len(packed) == 12 + 12 * dims.n_audio_layer + 29 * dims.n_text_layer
        d = dims.n_audio_state
        w1 = torch.from_numpy(sd["encoder.conv1.weight"])                     # [out, in, 3] -> [out, 3 * in] tap-major
        assert torch.equal(packed[0], w1.permute(0, 2, 1).reshape(d, -1).half())
        assert packed[4].dtype == torch.float32 and packed[4].shape == (dims.n_audio_ctx, d)       # sinusoids stay fp32
        enc0 = packed[12:24]
        q, k, v = (torch.from_numpy(sd[f"encoder.blocks.0.attn.{n}.weight"]).half() for n in ("query", "key", "value"))
        assert torch.equal(enc0[2], torch.cat([q, k, v], 0)) and enc0[0].dtype == torch.float32
        bias = enc0[3]
        assert torch.equal(bias[:d], torch.from_numpy(sd["encoder.blocks.0.attn.query.bias"]).half())
        assert float(bias[d: 2 * d].abs().max()) == 0.0                       # key has no bias (model.py:88)
        dec0 = packed[12 + 12 * dims.n_audio_layer: 12 + 12 * dims.n_audio_layer + 29]
        # LayerNorm folded into its consumer (csrc/dec_layer.cu): y = rstd * (x wf^T - mean * c1) + c2 == LN(x) W^T + b
        g = torch.from_numpy(sd["decoder.blocks.0.mlp_ln.weight"]).double()
        beta = torch.from_numpy(sd["decoder.blocks.0.mlp_ln.bias"]).double()
        w = torch.from_numpy(sd["decoder.blocks.0.mlp.0.weight"]).double()
        b = torch.from_numpy(sd["decoder.blocks.0.mlp.0.bias"]).double()
        wf, c1, c2 = dec0[26], dec0[27], dec0[28]
        assert wf.dtype == torch.float16 and c1.dtype == torch.float32 and c2.dtype == torch.float32
        x = torch.randn(5, dims.n_text_state, dtype=torch.float64) * 3 + 0.7
        mean, var = x.mean(-1, keepdim=True), x.var(-1, unbiased=False, keepdim=True)
        rstd = 1.0 / torch.sqrt(var + 1e-5)
        ref = ((x - mean) * rstd * g + beta) @ w.T + b
        got = rstd * (x @ wf.double().T - mean * c1.double()) + c2.double()
        assert float((got - ref).abs().max()) < 2e-2 * float(ref.abs().max())       # only the 16-bit rounding of W * gamma
        assert torch.allclose(c1.double(), wf.double().sum(1), atol=1e-3)
        kv = torch.cat([torch.from_numpy(sd[f"decoder.blocks.0.cross_attn.{n}.weight"]).half() for n in ("key", "value")], 0)
        assert torch.equal(dec0[10], kv) and dec0[10].shape == (2 * dims.n_text_state, dims.n_text_state)
        assert packed[7].dtype == torch.float16 and packed[8].dtype == torch.float32               # tied embedding, both types
        assert torch.equal(packed[8], torch.from_numpy(sd["decoder.token_embedding.weight"]).float())


class _FakeSession:
    """Stands in for decoding.DecoderSession: 'decodes' each audio to tokens that are a pure function of its
    features and prompt, stops after a per-session number of steps, and keeps beam-style finished stores."""
    log = []

    def __init__(self, task, n_audio):
        self.task, self.n_audio, self.G = task, n_audio, task.n_group
        self.temperature, self.seed = 0.0, None

    def set_audio(self, feats):
        self.key = [int(abs(float(f.sum())) * 10) % 50 for f in feats]

    def set_sampling(self, temperature, seed):
        self.temperature, self.seed = temperature, seed

    def prefill(self, init):
        self.init = np.asarray(init)

    def select(self):
        pass

    def run(self, max_steps):
        self.steps = 3 + (self.n_audio % 4)             # sessions of different size stop at different lengths
        _FakeSession.log.append((self.n_audio, self.seed))
        return self.steps

    def get(self, what):
        eot = self.task.tokenizer.eot
        n_init = self.init.shape[1]
        L = n_init + self.steps
        R = self.n_audio * self.G
        if what == "length":
            return torch.tensor([L])
        if what == "tokens":
            t = np.full((R, 448), eot, dtype=np.int32)
            for a in range(self.n_audio):
                for j in range(self.G):
                    t[a * self.G + j, :n_init] = self.init[a]
                    body = [1000 + self.key[a], 2000 + j, 3000 + int(self.init[a, -1]) % 7]
                    t[a * self.G + j, n_init: n_init + 3] = body
            return torch.from_numpy(t)
        if what == "sum_logprobs":
            return torch.tensor([-(1.0 + 0.1 * j + 0.01 * self.key[a]) for a in range(self.n_audio) for j in range(self.G)])
        if what == "no_speech":
            return torch.tensor([0.01 * self.key[a] for a in range(self.n_audio)])
        mc = max(1, round((self.task.options.beam_size or 1) * (self.task.options.patience or 1.0)))
        if what == "fin_tokens":
            t = np.full((self.n_audio, mc, 448), eot, dtype=np.int32)
            for a in range(self.n_audio):
                t[a, 0, : n_init + 2] = list(self.init[a]) + [1500 + self.key[a], eot]
            return torch.from_numpy(t)
        if what == "fin_len":
            return torch.from_numpy(np.tile(np.array([n_init + 2] + [0] * (mc - 1), dtype=np.int32), (self.n_audio, 1)))
        if what == "fin_score":
            return torch.from_numpy(np.tile(np.array([-0.5] + [0.0] * (mc - 1), dtype=np.float32), (self.n_audio, 1)))
        if what == "fin_count":
            return torch.ones(self.n_audio, dtype=torch.int32)
        raise KeyError(what)

    def close(self):
        pass


@pytest.mark.parametrize("opts", [dict(), dict(beam_size=3), dict(temperature=0.5, best_of=2, seed=9)])
def test_decoding_task_run_host_logic(opts, monkeypatch):
    """DecodingTask.run's host logic around the device session - per-row prompts, result assembly, ranking - with a
    fake session."""
    import contextlib

    import whisper_b200.decoding as WD

    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(WD.DecodingTask, "open_session", lambda self, n: _FakeSession(self, n))
    model = fake_model("test-en")
    feats = torch.arange(7 * 4 * 3, dtype=torch.float32).reshape(7, 4, 3) * 0.37
    monkeypatch.setattr(WD.DecodingTask, "_get_audio_features", lambda self, mel: mel)
    prompts = np.asarray([[50257, 50362 + (a % 3)] for a in range(7)], dtype=np.int32)
    _FakeSession.log = []
    task = WD.DecodingTask(model, WD.DecodingOptions(language="en", without_timestamps=True, **opts))
    init = np.tile(np.asarray(task.initial_tokens, dtype=np.int32), (7, 1))
    init[:, -1] = prompts[:, 1]
    res = task.run(feats, initial_tokens=init)
    assert len(res) == 7 and _FakeSession.log[0][0] == 7 and len(_FakeSession.log) == 1
    assert all(np.isfinite(r.avg_logprob) for r in res)


def test_official_checkpoint_table_and_sha256_gate(tmp_path):
    """load_model(<official name>) only accepts the cached file the reference would accept: right file name, SHA-256 equal
    to the digest in the reference's download URL (whisper/__init__.py:17-32, 63-71); the alignment-head dumps are the
    reference's (:36-51)."""
    import base64
    import gzip

    import whisper_b200 as wb

    table = wb._checkpoint_table()
    assert set(table) == {n for n in wb.available_models()}
    assert table["turbo"]["file"] == "large-v3-turbo.pt" and table["large"]["file"] == "large-v3.pt"
    assert all(len(e["sha256"]) == 64 and int(e["sha256"], 16) >= 0 for e in table.values())
    # every dump decodes to an (n_text_layer x n_text_head) mask with at least one head (model.py:278-285)
    for name, e in table.items():
        if e["alignment_heads"]:
            d = wb.dims_dict(name)
            mask = np.frombuffer(gzip.decompress(base64.b85decode(e["alignment_heads"].encode())), dtype=bool)
            assert mask.size == d["n_text_layer"] * d["n_text_head"] and mask.any()
    # the table IS the reference's (its _MODELS / _ALIGNMENT_HEADS, stored by oracle/make_golden.py: gen_checkpoints)
    with open(os.path.join(GOLD, "checkpoints_reference.json")) as f:
        ref = json.load(f)
    assert set(ref) == set(table)
    for name, e in ref.items():
        assert table[name]["file"] == os.path.basename(e["url"]) and table[name]["sha256"] == e["url"].split("/")[-2]
        assert table[name]["alignment_heads"] == e["alignment_heads"]
    # a file under the official name with other contents is refused before anything touches the GPU
    (tmp_path / "tiny.en.pt").write_bytes(b"not the official checkpoint")
    with pytest.raises(RuntimeError, match="SHA256"):
        wb.load_model("tiny.en", download_root=str(tmp_path))
    # no file and no synthetic weights: the reference would download; here it is an error that says so
    with pytest.raises(RuntimeError, match="no network"):
        wb.load_model("base.en", download_root=str(tmp_path))
    assert wb._resolve_official("base.en", str(tmp_path)) is None
