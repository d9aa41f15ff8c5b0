"""Generate the golden fixtures under tests/golden/ by RUNNING THE REFERENCE (openai/whisper,
imported read-only from /root/reference) on deterministic synthetic weights and audio.

    python -m oracle.make_golden            # from the repo root, in the build container

The reference cannot travel to the GPU box, so its outputs are committed as small fixtures; the
script is committed so they can be regenerated and audited.  Nothing is copied from the reference
except DATA it ships or computes: the mel filterbank asset, integer token-id tables, and its
numerical outputs on our inputs.

Fixtures:
  mel_filters.npz          whisper/assets/mel_filters.npz re-saved (audio.py:91-107)
  token_ids.json           special ids, non-speech suppress lists, " " encoding, language codes
  timing.npz               median_filter / dtw_cpu outputs (timing.py:19-105) on seeded inputs
  mel_<kind>.npz           log_mel_spectrogram outputs (sub-sampled) + global statistics
  alignment_<name>.npz     find_alignment tensor part: alignment matrix, DTW path, token probabilities
  model_<name>.npz/.json   encoder features (sub-sampled), prefill logits probes, and decode()
                           results (tokens, avg_logprob, no_speech_prob) for several DecodingOptions
  decode_extra_<name>.json decode() with task="translate", other language tokens, language=None and task="lang_id"
  checkpoints_reference.json  download URL and alignment-head dump per official model name
  state_dict_keys.json     names and shapes of the reference Whisper.state_dict() per architecture
  transcribe_<name>.json   whisper.transcribe() runs (transcribe.py:38-514) recorded as: every model.decode() call
                           the reference made (prompt, temperature, beam / best_of, a fingerprint of the window) with
                           its DecodingResult, every tokenizer.decode() text, and the final segments - enough to
                           replay the window loop (seek advance, prompt conditioning, temperature fallback,
                           no-speech skip, segment splitting) without a model
"""
from __future__ import annotations

import json
import os
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("WHISPER_REFERENCE", "/root/reference")
GOLD = os.path.join(REPO, "tests", "golden")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)

import whisper  # noqa: E402  (the reference)
from whisper.audio import log_mel_spectrogram, mel_filters  # noqa: E402
from whisper.decoding import DecodingOptions  # noqa: E402
from whisper.model import ModelDimensions, Whisper  # noqa: E402
from whisper.timing import dtw_cpu, median_filter  # noqa: E402
from whisper.tokenizer import LANGUAGES, get_tokenizer  # noqa: E402

from whisper_b200 import synthetic  # noqa: E402

# decode cases: name -> (DecodingOptions kwargs, n_audio)
DECODE_CASES = {
    "greedy": (dict(sample_len=48), 2),
    "greedy_notimestamps": (dict(sample_len=48, without_timestamps=True), 2),
    "greedy_prompt": (dict(sample_len=24, prompt=[1000 + 7 * i for i in range(40)]), 1),
    "greedy_prefix": (dict(sample_len=24, prefix=[2000 + 3 * i for i in range(5)]), 1),
    "greedy_nosuppress": (dict(sample_len=24, suppress_tokens="", suppress_blank=False), 1),
    "beam5": (dict(sample_len=40, beam_size=5), 2),
    "beam5_patience2": (dict(sample_len=40, beam_size=5, patience=2.0), 1),
    "beam3_lenpen": (dict(sample_len=32, beam_size=3, length_penalty=0.6), 1),
    "beam2_notimestamps": (dict(sample_len=32, beam_size=2, without_timestamps=True), 1),
}
FULL_LENGTH_CASE = ("greedy_full", dict(), 1)   # default sample_len = 224


# weight-generator settings per fixture model: "confident" = heavy-tailed logits (large top-1/top-2
# margins, the regime of a trained model); "diverse" = Gaussian logits (many near-ties, EOT and
# timestamp events everywhere - the hard case for selection logic)
SYNTH = {
    "confident": dict(),
    "diverse": dict(row_sigma=0.0, eot_scale=2.5, timestamp_scale=1.3),
    # "peaked" = even heavier-tailed token-embedding norms: beam candidates are separated by far more than 16-bit
    # activation noise (checked with the 16-bit emulation of oracle/model.py: the fp16-rounded trajectory of
    # beam5 equals the fp32 one for every step), so FREE-RUNNING beam search can be asserted step by step on the GPU
    "peaked": dict(row_sigma=1.0),
}
PEAKED_CASES = {
    "beam5": (dict(sample_len=24, beam_size=5), 2),
    "beam5_patience2": (dict(sample_len=24, beam_size=5, patience=2.0), 1),
    "beam3_lenpen": (dict(sample_len=24, beam_size=3, length_penalty=0.6), 1),
    "greedy": (dict(sample_len=24), 2),
}


def build_reference_model(name: str, seed: int, regime: str):
    dims = synthetic.dims_dict({"test-peak": "test-en"}.get(name, name))
    sd = synthetic.synthetic_state_dict(dims, seed=seed, **SYNTH[regime])
    model = Whisper(ModelDimensions(**dims))
    missing = model.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return model.eval(), dims


def gen_static():
    os.makedirs(GOLD, exist_ok=True)
    np.savez_compressed(os.path.join(GOLD, "mel_filters.npz"),
                        mel_80=mel_filters("cpu", 80).numpy(), mel_128=mel_filters("cpu", 128).numpy())
    from whisper.tokenizer import TO_LANGUAGE_CODE

    table = {"languages": list(LANGUAGES.keys()), "language_names": dict(TO_LANGUAGE_CODE)}   # tokenizer.py:10-128
    for key, multilingual, nl in (("gpt2", False, 99), ("multilingual", True, 99)):
        tok = get_tokenizer(multilingual, num_languages=nl, language="en", task="transcribe")
        table[key] = {"non_speech_tokens": list(tok.non_speech_tokens), "blank": tok.encode(" ")}
    specials = {}
    for n_vocab, multilingual, nl in ((51864, False, 99), (51865, True, 99), (51866, True, 100)):
        tok = get_tokenizer(multilingual, num_languages=nl, language="en", task="transcribe")
        specials[str(n_vocab)] = dict(
            eot=tok.eot, sot=tok.sot, translate=tok.translate, transcribe=tok.transcribe,
            sot_lm=tok.sot_lm, sot_prev=tok.sot_prev, no_speech=tok.no_speech,
            no_timestamps=tok.no_timestamps, timestamp_begin=tok.timestamp_begin,
            sot_sequence=list(tok.sot_sequence), all_language_tokens=list(tok.all_language_tokens),
            n_non_speech=len(tok.non_speech_tokens))
    table["specials"] = specials
    with open(os.path.join(GOLD, "token_ids.json"), "w") as f:
        json.dump(table, f)


def gen_timing():
    rng = np.random.Generator(np.random.PCG64(7))
    out = {}
    for i, shape in enumerate([(10,), (1, 15), (4, 5, 345), (3, 7, 1500)]):       # tests/test_timing.py:14-19
        x = rng.standard_normal(shape).astype(np.float32)
        out[f"med_in_{i}"] = x
        for w in (3, 5, 7, 13):                                                  # tests/test_timing.py:71
            out[f"med_out_{i}_{w}"] = median_filter(torch.from_numpy(x), w).numpy()
    for i, (N, M) in enumerate([(10, 20), (32, 16), (123, 1500), (234, 189)]):    # tests/test_timing.py:8-13
        x = rng.standard_normal((N, M)).astype(np.float32)
        out[f"dtw_in_{i}"] = x
        out[f"dtw_out_{i}"] = dtw_cpu(x.astype(np.float64)).astype(np.int32)
    np.savez_compressed(os.path.join(GOLD, "timing.npz"), **out)


def gen_mel():
    for kind in ("noise", "speechlike"):
        audio = synthetic.synthetic_audio(2, 480000, seed=1234, kind=kind)
        out = {}
        for n_mels in (80, 128):
            batch = log_mel_spectrogram(torch.from_numpy(audio), n_mels=n_mels).numpy()   # global max over batch
            single = log_mel_spectrogram(torch.from_numpy(audio[1, :160000]), n_mels=n_mels,
                                         padding=480000).numpy()                           # transcribe.py:139 usage
            out[f"batch_{n_mels}"] = batch[:, :, ::8].astype(np.float32)                  # every 8th frame
            out[f"batch_{n_mels}_head"] = batch[:, :, :64]
            out[f"batch_{n_mels}_tail"] = batch[:, :, -64:]
            out[f"single_{n_mels}"] = single[:, ::8]
            out[f"single_{n_mels}_shape"] = np.array(single.shape)
            out[f"batch_{n_mels}_sum"] = np.array([batch.astype(np.float64).sum(), batch.max(), batch.min()])
        np.savez_compressed(os.path.join(GOLD, f"mel_{kind}.npz"), **out)


def decode_case(model, mel, opts, n_audio):
    beam = opts.get("beam_size")
    options = DecodingOptions(language="en", fp16=False, temperature=0.0, **opts)
    results = []
    if beam:                      # reference raises for beam search with n_audio > 1 (decoding.py:734,740)
        for a in range(n_audio):
            results.append(model.decode(mel[a], options))
    else:
        results = model.decode(mel[:n_audio], options)
    return [dict(tokens=list(map(int, r.tokens)), avg_logprob=float(r.avg_logprob),
                 no_speech_prob=float(r.no_speech_prob)) for r in results]


def gen_model(name: str, seed: int, audio_kind: str, full_length: bool, regime: str, cases=None):
    t0 = time.time()
    model, dims = build_reference_model(name, seed, regime)
    audio = synthetic.synthetic_audio(2, 480000, seed=4321, kind=audio_kind)
    with torch.no_grad():
        mel = torch.stack([log_mel_spectrogram(torch.from_numpy(a), n_mels=dims["n_mels"]) for a in audio])
        feats = model.encoder(mel)
        tok = get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en",
                            task="transcribe")
        init = torch.tensor([list(tok.sot_sequence)] * 2)
        logits0 = model.decoder(init, feats)                       # prefill, all positions (model.py:245)
    arrays = {
        "feats_sub": feats[:, ::25, :].numpy(),                   # 60 of 1500 positions
        "feats_stats": np.array([float(feats.mean()), float(feats.std()), float(feats.abs().max())]),
        "logits0_last_top_idx": logits0[:, -1].topk(16).indices.numpy(),
        "logits0_last_top_val": logits0[:, -1].topk(16).values.numpy(),
        "logits0_last_sub": logits0[:, -1, ::97].numpy(),
        "logits0_sot_sub": logits0[:, 0, ::97].numpy(),
    }
    meta = {"name": name, "seed": seed, "audio_seed": 4321, "audio_kind": audio_kind, "dims": dims,
            "regime": regime, "synth_kwargs": SYNTH[regime], "decode": {}}
    cases = dict(DECODE_CASES if cases is None else cases)
    if full_length:
        cases[FULL_LENGTH_CASE[0]] = (FULL_LENGTH_CASE[1], FULL_LENGTH_CASE[2])
    for cname, (opts, n_audio) in cases.items():
        meta["decode"][cname] = {"options": opts, "n_audio": n_audio,
                                 "results": decode_case(model, mel, opts, n_audio)}
        print(f"  {name}/{cname}: {[len(r['tokens']) for r in meta['decode'][cname]['results']]} tokens "
              f"({time.time() - t0:.1f}s)", flush=True)
    if model.is_multilingual:
        with torch.no_grad():
            lang_tokens, lang_probs = model.detect_language(feats)
        meta["detect_language"] = {"tokens": lang_tokens.tolist(),
                                   "top": [max(p, key=p.get) for p in lang_probs],
                                   "top_prob": [max(p.values()) for p in lang_probs]}
    np.savez_compressed(os.path.join(GOLD, f"model_{name}.npz"), **arrays)
    with open(os.path.join(GOLD, f"model_{name}.json"), "w") as f:
        json.dump(meta, f)


def gen_alignment(name: str, seed: int, regime: str):
    """The tensor part of find_alignment (timing.py:176-216) executed with the reference's own model,
    hooks, median_filter and dtw on a fixed token row; word splitting (BPE strings) is left out."""
    from whisper.model import disable_sdpa
    from whisper.timing import dtw as ref_dtw

    model, dims = build_reference_model(name, seed, regime)
    audio = synthetic.synthetic_audio(1, 480000, seed=4321, kind="speechlike")
    tok = get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en", task="transcribe")
    rng = np.random.Generator(np.random.PCG64(99))
    text_tokens = [int(t) for t in rng.integers(1000, 40000, size=37)]
    num_frames = 2400
    with torch.no_grad():
        mel = log_mel_spectrogram(torch.from_numpy(audio[0]), n_mels=dims["n_mels"])
        tokens = torch.tensor([*tok.sot_sequence, tok.no_timestamps, *text_tokens, tok.eot])
        QKs = [None] * model.dims.n_text_layer
        hooks = [blk.cross_attn.register_forward_hook(lambda _, ins, outs, index=i: QKs.__setitem__(index, outs[-1][0]))
                 for i, blk in enumerate(model.decoder.blocks)]
        with disable_sdpa():
            logits = model(mel.unsqueeze(0), tokens.unsqueeze(0))[0]
        for h in hooks:
            h.remove()
        sampled = logits[len(tok.sot_sequence):, : tok.eot]
        probs = sampled.softmax(dim=-1)[np.arange(len(text_tokens)), text_tokens]
        heads = model.alignment_heads.indices().T
        weights = torch.stack([QKs[_l][_h] for _l, _h in heads])
        weights = weights[:, :, : num_frames // 2]
        weights = weights.softmax(dim=-1)
        std, mean = torch.std_mean(weights, dim=-2, keepdim=True, unbiased=False)
        weights = (weights - mean) / std
        weights = median_filter(weights, 7)
        matrix = weights.mean(axis=0)
        matrix = matrix[len(tok.sot_sequence): -1]
        text_idx, time_idx = ref_dtw(-matrix)
    np.savez_compressed(os.path.join(GOLD, f"alignment_{name}.npz"), text_tokens=np.array(text_tokens),
                        num_frames=np.array(num_frames), heads=heads.numpy(), matrix=matrix.numpy().astype(np.float32),
                        text_indices=np.asarray(text_idx), time_indices=np.asarray(time_idx),
                        token_probs=probs.numpy().astype(np.float32), seed=np.array(seed))


TRANSCRIBE_CASES = {
    # name -> (seconds of audio, audio kind, transcribe kwargs); thresholds are placed inside the range the
    # synthetic model produces (avg_logprob -0.7 .. -0.35, compression ratio 1.1 .. 1.8, no_speech_prob ~ 0) so that
    # some windows pass, some fall back to a sampled rung and some are skipped as silence
    "ladder_conditioned": (83, "speechlike", dict(sample_len=40, logprob_threshold=-0.45)),
    "ladder_compression": (70, "speechlike", dict(sample_len=40, compression_ratio_threshold=1.6,
                                                  temperature=(0.0, 0.6, 1.0))),
    "greedy_unconditioned": (64, "noise", dict(temperature=0.0, condition_on_previous_text=False, sample_len=32)),
    "beam_clips": (95, "speechlike", dict(temperature=(0.0, 0.4), beam_size=3, best_of=2, sample_len=28,
                                          clip_timestamps=[4.0, 41.5, 50.0], logprob_threshold=-0.43)),
    "silence_skip": (76, "noise", dict(temperature=(0.0, 0.4), no_speech_threshold=-1.0, logprob_threshold=-0.62,
                                       sample_len=32)),
    "no_thresholds": (47, "noise", dict(temperature=0.0, sample_len=36, no_speech_threshold=None,
                                        logprob_threshold=None, compression_ratio_threshold=None)),
}


def gen_transcribe(name: str, seed: int, regime: str):
    """Run the reference's transcribe() on synthetic weights / audio and record what its window loop did."""
    import importlib

    ref_tr = importlib.import_module("whisper.transcribe")     # the package attribute of that name is the function

    model, dims = build_reference_model(name, seed, regime)
    out = {"model": name, "seed": seed, "regime": regime, "cases": {}}
    for case, (secs, kind, kw) in TRANSCRIBE_CASES.items():
        audio = synthetic.synthetic_audio(1, 16000 * secs, seed=900 + secs, kind=kind)[0]
        calls, texts = [], {}
        orig_decode = model.decode

        def rec_decode(segment, options, _calls=calls, _orig=orig_decode):
            r = _orig(segment, options)
            _calls.append(dict(
                prompt=list(options.prompt or []), temperature=float(options.temperature),
                beam_size=options.beam_size, best_of=options.best_of, patience=options.patience,
                sample_len=options.sample_len,
                window_sum=float(segment.double().sum()), window_abs=float(segment.double().abs().sum()),
                tokens=list(r.tokens), avg_logprob=float(r.avg_logprob), no_speech_prob=float(r.no_speech_prob),
                compression_ratio=float(r.compression_ratio), result_temperature=float(r.temperature)))
            return r

        tok = get_tokenizer(model.is_multilingual, num_languages=model.num_languages, language="en", task="transcribe")
        orig_tok_decode = tok.decode

        def rec_tok_decode(token_ids, *a, _texts=texts, _orig=orig_tok_decode, **k):
            t = _orig(token_ids, *a, **k)
            _texts[",".join(str(int(x)) for x in token_ids)] = t
            return t

        tok.decode = rec_tok_decode              # get_tokenizer is lru_cached: transcribe() gets this same object
        model.decode = rec_decode
        torch.manual_seed(1234)
        try:
            result = ref_tr.transcribe(model, audio, verbose=None, fp16=False, language="en", **kw)
        finally:
            model.decode = orig_decode
            tok.decode = orig_tok_decode
        segs = [dict(id=sg["id"], seek=sg["seek"], start=sg["start"], end=sg["end"], text=sg["text"],
                     tokens=list(sg["tokens"]), temperature=sg["temperature"], avg_logprob=sg["avg_logprob"],
                     compression_ratio=sg["compression_ratio"], no_speech_prob=sg["no_speech_prob"])
                for sg in result["segments"]]
        out["cases"][case] = dict(seconds=secs, audio_kind=kind, audio_seed=900 + secs, kwargs=kw, calls=calls,
                                  texts=texts, segments=segs, text=result["text"], language=result["language"])
        print(f"transcribe {name}/{case}: {len(calls)} decode calls, {len(segs)} segments, "
              f"temperatures {sorted({c['temperature'] for c in calls})}")
    with open(os.path.join(GOLD, f"transcribe_{name}.json"), "w") as f:
        json.dump(out, f)


EXTRA_DECODE_CASES = {
    # name -> (DecodingOptions kwargs incl. language / task, n_audio); results are per audio
    "translate": (dict(language="en", task="translate", sample_len=32), 2),
    "translate_de_beam": (dict(language="de", task="translate", beam_size=3, sample_len=24), 1),
    "auto_language": (dict(language=None, sample_len=24), 2),
    "auto_language_beam": (dict(language=None, beam_size=2, sample_len=20), 2),
    "lang_id": (dict(language=None, task="lang_id"), 2),
    "french_prompt": (dict(language="fr", sample_len=20, prompt=[900 + 11 * i for i in range(9)]), 1),
}


def gen_decode_extra(name: str, seed: int, audio_kind: str, regime: str):
    """decode() with the task / language options the main fixture leaves at their defaults: translate, another
    language token, language=None (detect_language inside decode, decoding.py:666-678) and task="lang_id"."""
    model, dims = build_reference_model(name, seed, regime)
    audio = synthetic.synthetic_audio(2, 480000, seed=4321, kind=audio_kind)
    with torch.no_grad():
        mel = torch.stack([log_mel_spectrogram(torch.from_numpy(a), n_mels=dims["n_mels"]) for a in audio])
    out = {"name": name, "seed": seed, "audio_seed": 4321, "audio_kind": audio_kind, "regime": regime, "cases": {}}
    for cname, (opts, n_audio) in EXTRA_DECODE_CASES.items():
        options = DecodingOptions(fp16=False, temperature=0.0, **opts)
        with torch.no_grad():
            if opts.get("beam_size"):          # the reference cannot batch beam search (decoding.py:734,740)
                results = [model.decode(mel[a], options) for a in range(n_audio)]
            else:
                results = model.decode(mel[:n_audio], options)
        out["cases"][cname] = {"options": opts, "n_audio": n_audio, "results": [
            dict(tokens=list(map(int, r.tokens)), language=r.language,
                 avg_logprob=None if np.isnan(r.avg_logprob) else float(r.avg_logprob),
                 no_speech_prob=None if np.isnan(r.no_speech_prob) else float(r.no_speech_prob),
                 top_language_prob=None if r.language_probs is None else float(max(r.language_probs.values())))
            for r in results]}
        print(f"  {name}/{cname}: languages {[r.language for r in results]}, {[len(r.tokens) for r in results]} tokens")
    with open(os.path.join(GOLD, f"decode_extra_{name}.json"), "w") as f:
        json.dump(out, f)


def gen_state_dict_keys():
    """Names and shapes of the reference model's state dict (what a released checkpoint holds, __init__.py:147-156)
    for every architecture, built on the meta device so that large-v3 costs nothing."""
    out = {}
    for name in ("tiny.en", "tiny", "small", "large-v3", "large-v3-turbo", "test-en", "test-multi"):
        dims = synthetic.dims_dict(name)
        to_sparse = torch.Tensor.to_sparse           # the alignment-head buffer (non-persistent) has no meta kernel
        torch.Tensor.to_sparse = lambda self, *a, **k: self
        try:
            with torch.device("meta"):
                model = Whisper(ModelDimensions(**dims))
        finally:
            torch.Tensor.to_sparse = to_sparse
        out[name] = {k: list(v.shape) for k, v in model.state_dict().items()}
    with open(os.path.join(GOLD, "state_dict_keys.json"), "w") as f:
        json.dump(out, f)
    print("state dict keys:", {k: len(v) for k, v in out.items()})


def gen_checkpoints():
    """Per official model name: the reference's download URL (its last two components are the cached file's SHA-256
    and name, __init__.py:17-32) and its alignment-head dump (:36-51)."""
    out = {name: {"url": url, "alignment_heads": whisper._ALIGNMENT_HEADS[name].decode()
                  if name in whisper._ALIGNMENT_HEADS else None}
           for name, url in whisper._MODELS.items()}
    with open(os.path.join(GOLD, "checkpoints_reference.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("checkpoints:", len(out))


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    if sys.argv[1:] == ["test-peak"]:        # only the round-2 fixture (the others are unchanged since round 1)
        gen_model("test-peak", seed=21, audio_kind="speechlike", full_length=False, regime="peaked", cases=PEAKED_CASES)
        return
    if sys.argv[1:] == ["checkpoints"]:
        gen_checkpoints()
        return
    gen_static()
    gen_timing()
    gen_mel()
    gen_model("test-en", seed=11, audio_kind="speechlike", full_length=True, regime="confident")
    gen_model("test-multi", seed=12, audio_kind="noise", full_length=True, regime="diverse")
    gen_model("tiny.en", seed=13, audio_kind="speechlike", full_length=False, regime="confident")
    gen_model("test-peak", seed=21, audio_kind="speechlike", full_length=False, regime="peaked", cases=PEAKED_CASES)
    gen_alignment("test-en", seed=11, regime="confident")
    gen_transcribe("test-multi", seed=12, regime="diverse")
    gen_state_dict_keys()
    gen_decode_extra("test-multi", seed=12, audio_kind="noise", regime="diverse")
    gen_checkpoints()
    print("golden fixtures written to", GOLD)


if __name__ == "__main__":
    main()
