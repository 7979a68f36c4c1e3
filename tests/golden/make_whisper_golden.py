"""Golden vectors from the REFERENCE'S OWN Whisper model code (stt/models/whisper/whisper.py: AudioEncoder, TextDecoder with
its kv-cache protocol), executed in float64 with NumPy standing in for MLX (numpy_mlx_nn.py).  Run from the repo root in the
build container:  python tests/golden/make_whisper_golden.py   ->  tests/golden/whisper_golden.npz"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import numpy_mlx_nn as shim          # noqa: E402
import synth_params                  # noqa: E402

REF = "/root/reference/mlx_audio"
mx, nn = shim.install(precise=True)
if "--replay" not in sys.argv:                                 # replaying a --live record needs no reference source
    for name, path in (("mlx_audio", REF), ("mlx_audio.stt", f"{REF}/stt"), ("mlx_audio.stt.models", f"{REF}/stt/models"),
                       ("mlx_audio.stt.models.whisper", f"{REF}/stt/models/whisper")):
        shim.stub_package(name, path)
    import types                          # noqa: E402
    for stub, names in (("mlx_audio.stt.utils", ("load_audio",)), ("huggingface_hub", ("snapshot_download",))):
        m = types.ModuleType(stub)
        for n in names:
            setattr(m, n, None)
        sys.modules[stub] = m
    import mlx_audio.dsp as _dsp          # noqa: E402  (the reference's dsp.py, through the shim)
    u = types.ModuleType("mlx_audio.utils")
    u.hanning, u.mel_filters, u.stft = _dsp.hanning, _dsp.mel_filters, _dsp.stft
    sys.modules["mlx_audio.utils"] = u
    from mlx_audio.stt.models.whisper import whisper as W     # noqa: E402

DIMS = dict(n_mels=80, n_audio_ctx=60, n_audio_state=64, n_audio_head=4, n_audio_layer=2, n_vocab=300, n_text_ctx=32, n_text_state=64,
            n_text_head=4, n_text_layer=2)


class StubTokenizer:
    """The attributes DecodingTask and its logit filters read (decoding.py:445-507, 349-442), on a 300-entry vocabulary laid out like
    Whisper's: text < eot < the special block < timestamps."""
    eot, sot, lang_en, transcribe, translate, sot_lm, sot_prev, no_speech, no_timestamps, timestamp_begin = 200, 201, 202, 203, 204, 205, 206, 207, 208, 209
    sot_sequence = (201, 202, 203)
    sot_sequence_including_notimestamps = (201, 202, 203, 208)
    language = "en"

    def encode(self, text):
        return [7] if text == " " else [10 + (ord(c) % 150) for c in text]

    def decode(self, tokens):
        return " ".join(str(t) for t in tokens)


def decode_cases(model, mel, out):
    """DecodingTask._main_loop (decoding.py:588-632) with GreedyDecoder(temperature 0) and the three logit filters, on the encoder
    features of the model above.  The decoder's last-layer bias of a few timestamp tokens is raised so that the timestamp rules
    (pairs, text-after-pair, initial-timestamp window, probability-mass rule) all fire within the 14 sampled tokens."""
    from mlx_audio.stt.models.whisper import decoding as D
    model.get_tokenizer = lambda language=None, task=None: StubTokenizer()
    gain = float(os.environ.get("TEXT_GAIN", "3.0"))                 # text rows of the tied embedding: makes text tokens competitive with the
    w = np.array(model.decoder.token_embedding.weight)              # summed timestamp mass, so that the mass rule fires on some steps only
    w[:StubTokenizer.eot] *= gain
    model.decoder.token_embedding.weight = mx.array(w)
    out["dec_text_gain"] = gain
    suppress = [3, 4, 5, 250]
    for tag, opts in (("ts", dict()), ("nots", dict(without_timestamps=True))):
        options = D.DecodingOptions(language="en", temperature=0.0, sample_len=14, suppress_tokens=suppress, fp16=False, **opts)
        task = D.DecodingTask(model, options)
        task.inference.reset()
        feats = task._get_audio_features(mx.array(mel))
        tokens = mx.broadcast_to(mx.array(task.initial_tokens), (mel.shape[0], len(task.initial_tokens)))
        tokens, sum_lp, no_speech = task._main_loop(feats, tokens)
        out[f"dec_{tag}_tokens"], out[f"dec_{tag}_sum_logprobs"], out[f"dec_{tag}_no_speech"] = np.asarray(tokens), np.asarray(sum_lp), np.asarray(no_speech)
        print(tag, np.asarray(tokens).tolist(), np.asarray(sum_lp))
        res = task.run(mx.array(mel))                                # the public result objects (decoding.py:634-722)
        out[f"dec_{tag}_run"] = json.dumps([dict(language=r.language, tokens=[int(t) for t in r.tokens], text=r.text, avg_logprob=float(r.avg_logprob),
                                                 no_speech_prob=float(r.no_speech_prob), temperature=float(r.temperature),
                                                 compression_ratio=float(r.compression_ratio)) for r in res])
    out["dec_suppress"] = np.asarray(suppress)
    # the three logit filters and GreedyDecoder.update applied directly to random logits under hand-built token histories
    tk = StubTokenizer()
    sb = 3
    filters = [D.SuppressBlank(tk, sb, 300), D.SuppressTokens(suppress, 300), D.ApplyTimestampRules(tk, sb, 2)]
    rng = np.random.default_rng(23)
    T, E = tk.timestamp_begin, tk.eot
    hist = {"first": [[]] * 3,
            "mixed": [[11, 12, 13], [11, 12, T + 5], [11, T + 4, T + 5], [T + 1, T + 1, 12], [T + 2, 12, T + 9], [11, 12, E], [T, T, 14], [11, T, T + 30]],
            "one": [[T + 3], [17], [T]], "two": [[T + 3, T + 3], [17, T + 8], [T + 1, 20]]}
    for name, rows in hist.items():
        toks = np.array([[201, 202, 203] + r for r in rows], dtype=np.int32)
        logits = 3.0 * rng.standard_normal((len(rows), 300))
        if name == "mixed":
            logits[0, T:] += 4.0                                     # row 0: timestamp mass beats every text token
        y = mx.array(logits)
        for f in filters:
            y = f.apply(y, mx.array(toks))
        dec = D.GreedyDecoder(0.0, E)
        nt, completed, slp = dec.update(mx.array(toks), y, mx.zeros(len(rows)))
        out[f"filt_{name}_tokens"], out[f"filt_{name}_logits"], out[f"filt_{name}_out"] = toks, logits, np.asarray(y)
        out[f"filt_{name}_next"], out[f"filt_{name}_sum_logprobs"], out[f"filt_{name}_completed"] = np.asarray(nt), np.asarray(slp), bool(completed)
    out["dec_max_initial_timestamp_index"] = round(1.0 / (30.0 / DIMS["n_audio_ctx"]))


GEN_DIMS = dict(n_mels=80, n_audio_ctx=1500, n_audio_state=32, n_audio_head=2, n_audio_layer=1, n_vocab=300, n_text_ctx=48, n_text_state=32,
                n_text_head=2, n_text_layer=2)


def generate_case(out):
    """Model.generate (whisper.py:799-1318) on 75 s of synthetic audio: three 30-second windows through decode_with_fallback (temperatures
    0 / 0.4 / 0.8 / 1.0), the no-speech skip, segment cutting at consecutive timestamp tokens, the seek rule, previous-text conditioning with
    the prompt reset after a hot window.  The model is tiny (one encoder layer of width 32) but keeps n_audio_ctx = 1500 so that the
    reference's hard-coded 3000-frame windows fit.  Categorical draws: D.categorical is replaced by the inverse-CDF draw of the stand-in fed
    from a table U[k, step], k = index of the decode call among those made at a temperature > 0 (one table row per call, so the
    reference's extra discarded step after completion does not shift later draws)."""
    from mlx_audio.stt.models.whisper import decoding as D
    sys.modules["mlx_audio.stt.utils"].merge_hotwords = lambda prompt, hotwords: prompt
    model = W.Model(W.ModelDimensions(**GEN_DIMS), dtype=mx.float32)
    names = [(n, v.shape) for n, v in shim.flat_parameters(model)]
    for n, sh in names:
        shim.set_parameter(model, n, synth_params.value(n, sh))
    model.get_tokenizer = lambda language=None, task=None: StubTokenizer()
    gain = 3.0
    w0 = np.array(model.decoder.token_embedding.weight)

    def set_gain(gv):
        w = w0.copy()
        w[:StubTokenizer.eot] *= gv
        model.decoder.token_embedding.weight = mx.array(w)
    set_gain(gain)
    rng = np.random.default_rng(33)
    sr = 16000
    t = np.arange(75 * sr) / sr
    audio = (0.2 * np.sin(2 * np.pi * 220 * t) * (1 + np.sin(2 * np.pi * 0.3 * t)) + 0.05 * rng.standard_normal(t.shape)).astype(np.float32)
    audio[int(31 * sr):int(58 * sr)] *= 1e-3                      # a quiet stretch
    U = rng.random((64, GEN_DIMS["n_text_ctx"] // 2 + 4))
    state = {"call": -1, "step": 0, "temps": []}
    run0 = D.DecodingTask.run

    def run(self, mel):
        state["temps"].append(float(self.options.temperature))
        if self.options.temperature > 0:
            state["call"] += 1
            state["step"] = 0
        return run0(self, mel)

    def cat(logits, temp):
        u = U[state["call"], state["step"]]
        state["step"] += 1
        mx.random.queue.append(("categorical", np.full(np.asarray(logits).shape[:-1], u)))
        return mx.random.categorical(logits / temp)
    D.DecodingTask.run, D.categorical = run, cat
    mx.random.strict = True
    cases = {"default": dict(temperature=(0.0, 0.4, 0.8, 1.0), logprob_threshold=-4.6, compression_ratio_threshold=2.4, no_speech_threshold=0.6),
             "nocond": dict(temperature=(0.0, 0.5), logprob_threshold=-4.3, condition_on_previous_text=False, no_speech_threshold=None,
                            initial_prompt_tokens=[11, 12, 13]),
             "nots": dict(temperature=0.0, return_timestamps=False, clip_timestamps="5,40"),
             # weaker text rows: the timestamp-mass rule fires after some text, which closes timestamp PAIRS -> segments cut at the pairs and
             # seek moves to the last closed timestamp instead of by a whole window
             "pairs": dict(temperature=(0.0, 0.6), logprob_threshold=-5.2, no_speech_threshold=None, clip_timestamps="0,9",
                           text_gain=float(os.environ.get("GEN_GAIN2", "1.6")))}
    try:
        for tag, kw in cases.items():
            state.update(call=-1, step=0, temps=[])
            kw = dict(kw)
            set_gain(kw.pop("text_gain", gain))
            prompt_tokens = kw.pop("initial_prompt_tokens", None)
            if prompt_tokens is not None:                           # the stub tokenizer's encode() ignores the text and returns these ids
                StubTokenizer.encode = lambda self, text, _p=prompt_tokens: list(_p)
                kw["initial_prompt"] = "x"
            res = model.generate(mx.array(audio), language="en", verbose=None, suppress_tokens=[3, 4, 5, 250], sample_len=14, fp16=False, **kw)
            segs = [{k: (v if not isinstance(v, (np.floating, np.integer)) else v.item()) for k, v in sg.items()} for sg in res.segments]
            for sg in segs:
                sg["tokens"] = [int(t_) for t_ in sg["tokens"]]
                sg.pop("words", None)
            out[f"gen_{tag}"] = json.dumps(dict(text=res.text, language=res.language, segments=segs, temps=state["temps"]))
            print(tag, "decode calls", len(state["temps"]), "hot", sum(t_ > 0 for t_ in state["temps"]), "segments", len(segs),
                  [(s_["seek"], round(s_["start"], 2), round(s_["end"], 2), len(s_["tokens"])) for s_ in segs[:8]])
    finally:
        D.DecodingTask.run = run0
        mx.random.strict = False
    out["gen_audio_head"], out["gen_U"], out["gen_text_gain"] = audio[:16], U, gain      # the audio is rebuilt from the formula above (seed 33)
    out["gen_pairs_gain"] = float(os.environ.get("GEN_GAIN2", "1.6"))
    out["gen_params"] = synth_params.manifest(names)
    out["gen_suppress"] = np.asarray([3, 4, 5, 250])


def main():
    model = W.Model(W.ModelDimensions(**DIMS), dtype=mx.float32)
    names = [(n, v.shape) for n, v in shim.flat_parameters(model)]
    for n, sh in names:
        shim.set_parameter(model, n, synth_params.value(n, sh))
    rng = np.random.default_rng(21)
    mel = rng.standard_normal((2, 2 * DIMS["n_audio_ctx"], DIMS["n_mels"]))
    xa = model.encoder(mx.array(mel))
    tokens = rng.integers(0, DIMS["n_vocab"], size=(2, 7))
    logits, kv, cross_qk = model.decoder(mx.array(tokens), xa)
    step_tokens = rng.integers(0, DIMS["n_vocab"], size=(2, 3))
    step_logits = []
    for i in range(step_tokens.shape[1]):
        lg, kv, _ = model.decoder(mx.array(step_tokens[:, i:i + 1]), xa, kv_cache=kv)
        step_logits.append(np.asarray(lg))
    out = dict(params=synth_params.manifest(names), mel=mel, xa=np.asarray(xa), tokens=tokens, logits=np.asarray(logits),
               cross_qk_last=np.asarray(cross_qk[-1]), step_tokens=step_tokens, step_logits=np.stack(step_logits, 1)[:, :, 0],
               sinusoids=np.asarray(W.sinusoids(60, 64)))
    decode_cases(model, mel, out)
    generate_case(out)
    np.savez_compressed(os.path.join(os.environ.get("GOLDEN_OUT", HERE), "whisper_golden.npz"), **out)
    print(len(out), "entries")


def live(n):
    """--live N: N random configurations, reference classes vs oracle/whisper.py, no fixture involved (tests/test_golden_reproducible.py)."""
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import whisper as OW
    from live_tape import Tape
    tape = Tape("whisper", n, sys.argv)
    worst = 0.0
    for seed in range(n):
        rng = np.random.default_rng(1000 + seed)
        heads = int(rng.choice([1, 2, 4]))
        state = heads * int(rng.choice([8, 16]))
        d = dict(n_mels=int(rng.choice([16, 80])), n_audio_ctx=int(rng.integers(5, 40)), n_audio_state=state, n_audio_head=heads,
                 n_audio_layer=int(rng.integers(1, 4)), n_vocab=int(rng.integers(50, 200)), n_text_ctx=int(rng.integers(8, 24)), n_text_state=state,
                 n_text_head=heads, n_text_layer=int(rng.integers(1, 4)))
        if tape.reference:
            model = W.Model(W.ModelDimensions(**d), dtype=mx.float32)
        names = tape.value(lambda: [(k, v.shape) for k, v in shim.flat_parameters(model)])
        if tape.reference:
            for k, sh in names:
                shim.set_parameter(model, k, synth_params.value(k, sh))
        P = {k: torch.as_tensor(synth_params.value(k, sh)) for k, sh in names}
        b = int(rng.integers(1, 4))
        mel = rng.standard_normal((b, 2 * d["n_audio_ctx"], d["n_mels"]))
        if tape.reference:
            xa = model.encoder(mx.array(mel))
        oxa = OW.encoder(P, torch.as_tensor(mel), d)
        nt = int(rng.integers(1, d["n_text_ctx"] - 3))
        toks = rng.integers(0, d["n_vocab"], size=(b, nt))
        if tape.reference:
            lg, kv, _ = model.decoder(mx.array(toks), xa)
        olg, cache = OW.decoder_forward(P, torch.as_tensor(toks), oxa, None, d)
        errs = [tape.err(lambda: xa, oxa.numpy()), tape.err(lambda: lg, olg.numpy())]
        for _ in range(2):
            t1 = rng.integers(0, d["n_vocab"], size=(b, 1))
            if tape.reference:
                lg, kv, _ = model.decoder(mx.array(t1), xa, kv_cache=kv)
            olg, cache = OW.decoder_forward(P, torch.as_tensor(t1), oxa, cache, d)
            errs.append(tape.err(lambda: lg, olg.numpy()))
        worst = max(worst, float(max(errs)))
        print("whisper", d, "max err", float(max(errs)))
    # logit filters + greedy update on random logits under random token histories (decoding.py:307-442)
    if tape.reference:
        from mlx_audio.stt.models.whisper import decoding as D
    tk = StubTokenizer()
    spec = OW.TokenizerSpec(eot=200, sot=201, no_timestamps=208, timestamp_begin=209, no_speech=207, blank_ids=(7,), language=202, task=203,
                            transcribe=203, translate=204, sot_lm=205, sot_prev=206)
    T, E = tk.timestamp_begin, tk.eot
    cases = 40 * n
    for case in range(cases):
        rng = np.random.default_rng(7000 + case)
        B, L = int(rng.integers(1, 5)), int(rng.integers(0, 7))
        pool = np.concatenate([rng.integers(0, E, size=20), rng.integers(T, 300, size=20), [E, T, T + 1]])
        hist = rng.choice(pool, size=(B, L))
        toks = np.concatenate([np.tile([201, 202, 203], (B, 1)), hist], axis=1).astype(np.int32)
        logits = rng.standard_normal((B, 300)) * float(rng.choice([0.5, 3.0]))
        if rng.random() < 0.4:
            logits[:, T:] += float(rng.uniform(1, 6))
        sup = sorted(set(int(v) for v in rng.integers(0, 300, size=int(rng.integers(0, 6)))))
        mi = [None, 0, 2, 30][int(rng.integers(0, 4))]
        if tape.reference:
            filters = [D.SuppressBlank(tk, 3, 300)] + ([D.SuppressTokens(sup, 300)] if sup else []) + [D.ApplyTimestampRules(tk, 3, mi)]
            y = mx.array(logits)
            for f in filters:
                y = f.apply(y, mx.array(toks))
            y = np.asarray(y)
        want = OW.apply_filters(torch.as_tensor(logits), toks.tolist(), spec, 3, sup, max_initial_timestamp_index=mi).numpy()
        assert tape.err(lambda: y, want, same_nonfinite=True) < 1e-12, (case, toks.tolist(), sup, mi)
        if tape.reference:
            nt, comp, slp = D.GreedyDecoder(0.0, E).update(mx.array(toks), mx.array(y), mx.zeros(B))
        ont, ocomp, oslp = OW.greedy_update(toks.tolist(), torch.as_tensor(want), torch.zeros(B, dtype=torch.float64), E)
        nt, comp, slp = tape.value(lambda: (np.asarray(nt), bool(comp), np.asarray(slp, dtype=np.float64)))
        assert np.array_equal(np.asarray(nt), np.array(ont)) and comp == ocomp and np.allclose(np.asarray(slp), oslp.numpy(), rtol=0, atol=1e-12, equal_nan=True), case
    tape.close()
    print("filter / greedy cases identical:", cases)
    assert worst < 1e-10, worst
    print("LIVE OK", worst)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--live":
        live(int(sys.argv[2]))
    else:
        main()
