"""Golden vectors from the REFERENCE'S OWN Qwen3-TTS code (tts/models/qwen3_tts/{talker,speech_tokenizer,qwen3_tts}.py,
lm/models/cache.py, lm/sample_utils.py) executed in float64 with NumPy standing in for MLX (numpy_mlx_nn.py), at a reduced
configuration.  Run from the repo root in the build container:  python tests/golden/make_qwen3_golden.py
->  tests/golden/qwen3_golden.npz

``mx.random.categorical`` is not reproducible outside MLX, so here (as in oracle/qwen3.py and the CUDA sampler) the categorical
draw is the inverse CDF in index order driven by an injected uniform; everything around the draw is the reference's code."""
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import numpy_mlx_nn as shim          # noqa: E402
import synth_params                  # noqa: E402

REF = "/root/reference/mlx_audio"
mx, nn = shim.install(precise=True)
if "--replay" not in sys.argv:                                 # replaying a --live record needs no reference source
    for name, path in (("mlx_audio", REF), ("mlx_audio.lm", f"{REF}/lm"), ("mlx_audio.lm.models", f"{REF}/lm/models"), ("mlx_audio.tts", f"{REF}/tts"),
                       ("mlx_audio.tts.models", f"{REF}/tts/models"), ("mlx_audio.tts.models.qwen3_tts", f"{REF}/tts/models/qwen3_tts"),
                       ("mlx_audio.codec", f"{REF}/codec"), ("mlx_audio.codec.models", f"{REF}/codec/models"),
                       ("mlx_audio.codec.models.mimi", f"{REF}/codec/models/mimi")):
        shim.stub_package(name, path)
    for stub, names in (("huggingface_hub", ("snapshot_download", "hf_hub_download")),):
        m = types.ModuleType(stub)
        for n in names:
            setattr(m, n, None)
        sys.modules[stub] = m
    u = types.ModuleType("mlx_audio.utils")
    u.load_audio = None
    import mlx_audio.dsp as _dsp          # noqa: E402
    u.hanning, u.mel_filters, u.stft = _dsp.hanning, _dsp.mel_filters, _dsp.stft
    sys.modules["mlx_audio.utils"] = u

    from mlx_audio.tts.models.qwen3_tts import config as C            # noqa: E402
    from mlx_audio.tts.models.qwen3_tts import talker as T            # noqa: E402

CP = dict(vocab_size=80, hidden_size=48, intermediate_size=96, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, head_dim=16,
          num_code_groups=4)
TALKER = dict(vocab_size=1104, hidden_size=64, intermediate_size=128, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
              head_dim=16, rope_scaling={"interleaved": True, "mrope_section": [2, 3, 3], "rope_type": "default"}, num_code_groups=4,
              text_hidden_size=40, text_vocab_size=120, codec_eos_token_id=1000, codec_pad_id=1001, codec_bos_id=1002, codec_think_id=1003,
              codec_nothink_id=1004, codec_think_bos_id=1005, codec_think_eos_id=1006, codec_language_id={"english": 1010, "german": 1011},
              spk_id={"amy": 1020, "bob": 1021}, code_predictor_config=CP)
ORACLE_CFG = {"vocab_size": 1104, "hidden_size": 64, "intermediate_size": 128, "num_hidden_layers": 2, "num_attention_heads": 4,
              "num_key_value_heads": 2, "head_dim": 16, "rms_norm_eps": 1e-6, "rope_theta": 1000000.0, "mrope_section": [2, 3, 3],
              "num_code_groups": 4, "codec_eos_token_id": 1000, "text_hidden_size": 40, "cp_vocab_size": 80, "cp_hidden_size": 48,
              "cp_intermediate_size": 96, "cp_num_hidden_layers": 2, "cp_num_attention_heads": 4, "cp_num_key_value_heads": 2, "cp_head_dim": 16,
              "cp_rope_theta": 1000000.0}


def fill(module, prefix="", rule=lambda name: None):
    names = [(prefix + n, v.shape, rule(n)) for n, v in shim.flat_parameters(module)]
    for n, sh, r in names:
        shim.set_parameter(module, n[len(prefix):], synth_params.value(n, sh, r))
    for m in module.modules():                                       # Mimi codebooks keep a derived embedding table
        if hasattr(m, "update_in_place"):
            m.update_in_place()
    return names


def talker_cases(out):
    talker = T.Qwen3TTSTalkerForConditionalGeneration(C.Qwen3TTSTalkerConfig(**TALKER))
    names = fill(talker)
    out["talker_params"] = synth_params.manifest(names)
    rng = np.random.default_rng(31)
    x = rng.standard_normal((2, 6, 64))
    cache = talker.make_cache()
    logits, hidden = talker(mx.array(x), cache=cache)
    out["t_x"], out["t_logits"], out["t_hidden"] = x, np.asarray(logits), np.asarray(hidden)
    xs = rng.standard_normal((2, 3, 64))
    sl = []
    for i in range(3):
        lg, hd = talker(mx.array(xs[:, i:i + 1]), cache=cache)
        sl.append(np.asarray(lg)[:, 0])
    out["t_step_x"], out["t_step_logits"] = xs, np.stack(sl, 1)
    # code predictor: 2-token prefill (hidden, code-0 embedding) then single-token steps, one lm_head per generation step
    cc = talker.code_predictor.make_cache()
    cx = rng.standard_normal((1, 2, 64))
    cl, cc, _ = talker.code_predictor(mx.array(cx), cache=cc, generation_step=0)
    cs = [np.asarray(cl)[:, -1]]
    cx2 = rng.standard_normal((1, 2, 64))
    for i in range(2):
        cl, cc, _ = talker.code_predictor(mx.array(cx2[:, i:i + 1]), cache=cc, generation_step=i + 1)
        cs.append(np.asarray(cl)[:, -1])
    out["cp_x"], out["cp_x2"], out["cp_logits"] = cx, cx2, np.stack(cs, 1)
    return talker


TOKDEC = dict(latent_dim=32, codebook_dim=16, codebook_size=80, decoder_dim=48, hidden_size=32, intermediate_size=64, head_dim=8,
              num_attention_heads=4, num_hidden_layers=2, num_key_value_heads=4, num_quantizers=4, num_semantic_quantizers=1, sliding_window=6,
              upsample_rates=[8, 5, 4, 3], upsampling_ratios=[2, 2])
ORACLE_TOK = {"latent_dim": 32, "codebook_dim": 16, "codebook_size": 80, "decoder_dim": 48, "hidden_size": 32, "intermediate_size": 64,
              "layer_scale_initial_scale": 0.01, "head_dim": 8, "num_attention_heads": 4, "num_hidden_layers": 2, "num_key_value_heads": 4,
              "num_quantizers": 4, "num_semantic_quantizers": 1, "rms_norm_eps": 1e-5, "rope_theta": 10000.0, "upsample_rates": [8, 5, 4, 3],
              "upsampling_ratios": [2, 2], "sliding_window": 6}


TOKENC = dict(hidden_size=32, num_filters=4, upsampling_ratios=[8, 6, 5, 4], intermediate_size=64, num_attention_heads=4, num_key_value_heads=4,
              num_hidden_layers=2, sliding_window=6, codebook_dim=16, codebook_size=64, num_quantizers=20, head_dim=8)
ORACLE_TOKENC = {"dimension": 32, "nfilters": 4, "ratios": [8, 6, 5, 4], "ksize": 7, "residual_ksize": 3, "last_ksize": 3, "compress": 2, "d_model": 32,
                 "num_heads": 4, "num_layers": 2, "dim_feedforward": 64, "context": 6, "max_period": 10000, "layer_scale": 0.01, "nq": 20, "bins": 64,
                 "qdim": 16, "upsample_stride": 2, "valid_num_quantizers": 16}


class CharTokenizer:
    """Stands in for the HF tokenizer: the three chat-template markers are single ids, every other character is one id."""
    MARK = {"<|im_start|>": 1, "<|im_end|>": 2, "assistant": 3, "user": 4, "\n": 5}

    def __init__(self):
        self.calls = []

    def encode(self, text):
        ids, i = [], 0
        while i < len(text):
            for m, v in self.MARK.items():
                if text.startswith(m, i):
                    ids.append(v)
                    i += len(m)
                    break
            else:
                ids.append(10 + (ord(text[i]) % 100))
                i += 1
        self.calls.append(ids)
        return ids


def tokenizer_cases(out):
    from mlx_audio.tts.models.qwen3_tts import speech_tokenizer as S
    tok = S.Qwen3TTSSpeechTokenizer(C.Qwen3TTSTokenizerConfig(decoder_config=C.Qwen3TTSTokenizerDecoderConfig(**TOKDEC),
                                                              encoder_config=C.Qwen3TTSTokenizerEncoderConfig(**TOKENC)))
    names = fill(tok, rule=lambda n: "small" if n.endswith((".alpha", ".beta")) else ("scale0.08" if n == "decoder.decoder.6.conv.weight" else None))     # SnakeBeta gains are exp(alpha), exp(beta)
    out["tok_params"] = synth_params.manifest(names)
    out["tok_cfg"] = json.dumps(ORACLE_TOK)
    out["tok_enc_cfg"] = json.dumps(ORACLE_TOKENC)
    rng = np.random.default_rng(33)
    codes = rng.integers(0, 80, size=(2, 4, 9))                    # [B, n_q, T]
    out["tok_codes"], out["tok_wav"] = codes, np.asarray(tok.decoder(mx.array(codes)))
    print("clipped fraction", float((np.abs(out["tok_wav"]) >= 1).mean()))
    out["tok_wav_chunked"] = np.asarray(tok.decoder.chunked_decode(mx.array(codes), chunk_size=4, left_context_size=2))
    codes_bt = rng.integers(0, 80, size=(2, 7, 4))                 # [B, T, n_q], public decode
    codes_bt[1, 5:, :] = 0                                         # trailing zero codes shorten the reported length
    wav, lens = tok.decode(mx.array(codes_bt))
    out["tok_codes_bt"], out["tok_decode_wav"], out["tok_decode_lens"] = codes_bt, np.asarray(wav), np.asarray(lens)
    # encoder (ICL voice cloning): audio -> the first 16 of 20 code books, 5 frames + 300 samples
    audio = 0.4 * np.random.default_rng(133).standard_normal((2, 1, 5 * 1920 + 300))      # regenerated by the test from the seed
    out["tok_enc_codes"] = np.asarray(tok.encode(mx.array(audio)))
    print("tokenizer encode", out["tok_enc_codes"].shape)
    # streaming decoder: two calls of new codes with conv buffers and the transformer kv cache
    tok.decoder.reset_streaming_state()
    parts = [np.asarray(tok.decoder.streaming_step(mx.array(codes[:1, :, :5]))), np.asarray(tok.decoder.streaming_step(mx.array(codes[:1, :, 5:])))]
    tok.decoder.reset_streaming_state()
    out["tok_stream_wav"] = np.concatenate(parts, axis=-1)
    return tok


def model_cases(out, tok):
    from mlx_audio.tts.models.qwen3_tts import qwen3_tts as Q
    cfg = C.ModelConfig(talker_config=dict(TALKER), tts_model_type="custom_voice", tts_pad_token_id=111, tts_bos_token_id=112, tts_eos_token_id=113)
    model = Q.Model(cfg)
    names = fill(model.talker)
    assert synth_params.manifest(names) == out["talker_params"]
    eos = TALKER["codec_eos_token_id"]
    gain = float(os.environ.get('EOS_GAIN', '2.0'))
    w = np.array(model.talker.codec_head.weight)
    w[eos] *= gain                                                  # makes EOS reachable within a few frames
    model.talker.codec_head.weight = mx.array(w)
    model.load_speech_tokenizer(tok)
    model.tokenizer = CharTokenizer()
    mx.random.strict = True
    captured = {}
    real_decode = tok.decode

    def spy(codes):
        captured["codes"] = np.asarray(codes)
        return real_decode(codes)
    tok.decode = spy
    out["gen_eos_gain"] = gain
    cases = [dict(tag="a", text="Hello there, world.", voice="Amy", instruct="calm", lang_code="english", max_tokens=40, seed=int(os.environ.get("SEED_A", "45"))),
             dict(tag="b", text="Short one", voice="bob", instruct=None, lang_code="auto", max_tokens=6, seed=42, top_p=0.8),
             dict(tag="c", text="Greedy decoding path", voice="amy", instruct=None, lang_code="german", max_tokens=5, seed=43, temperature=0.0)]
    for c in cases:
        g = TALKER["num_code_groups"]
        us = np.random.default_rng(c["seed"]).random((c["max_tokens"], g))
        greedy = c.get("temperature", 0.9) <= 0
        mx.random.queue[:] = [] if greedy else [("categorical", np.array([v])) for v in us.reshape(-1)]
        model.tokenizer.calls.clear()
        ie, tr, pad = model._prepare_generation_inputs(c["text"], language=c["lang_code"], speaker=c["voice"], instruct=c["instruct"])
        text_ids = model.tokenizer.calls[0]
        instruct_ids = model.tokenizer.calls[1] if c["instruct"] else None
        captured.clear()
        res = list(model.generate(text=c["text"], voice=c["voice"], instruct=c["instruct"], lang_code=c["lang_code"], max_tokens=c["max_tokens"],
                                  temperature=c.get("temperature", 0.9), top_p=c.get("top_p", 1.0)))
        t = c["tag"]
        out[f"gen_{t}_meta"] = json.dumps({k: v for k, v in c.items() if k != "seed"} | {"text_ids": text_ids, "instruct_ids": instruct_ids,
                                                                                         "draws_left": len(mx.random.queue)})
        out[f"gen_{t}_u"] = us
        out[f"gen_{t}_input_embeds"], out[f"gen_{t}_trailing"], out[f"gen_{t}_pad"] = np.asarray(ie), np.asarray(tr), np.asarray(pad)
        out[f"gen_{t}_codes"] = captured["codes"][0]
        out[f"gen_{t}_audio"] = np.asarray(res[0].audio)
        print(t, "frames", captured["codes"].shape, "audio", res[0].audio.shape, "draws left", len(mx.random.queue))
    mx.random.queue[:] = []
    # ---- batch path: Model.batch_generate's own loop (qwen3_tts.py:1800-1935; reached without ICL through stream=True, with a
    # streaming interval long enough that every sequence is decoded once, at the end) ----
    texts, voices, instructs = ["First line.", "The second one is longer", "Hi"], ["amy", "bob", "amy"], ["calm and slow", None, "sad"]
    max_tokens = int(os.environ.get("BATCH_MAX", "12"))
    g = TALKER["num_code_groups"]
    ub = np.random.default_rng(int(os.environ.get("SEED_B", "51"))).random((max_tokens, g, len(texts)))
    mx.random.queue[:] = [("categorical", ub[s, k]) for s in range(max_tokens) for k in range(g)]
    model.tokenizer.calls.clear()
    seen = []
    real_chunked = tok.decoder.chunked_decode

    def spy_chunked(codes, *a, **k):
        seen.append(np.asarray(codes))
        return real_chunked(codes, *a, **k)
    tok.decoder.chunked_decode = spy_chunked
    res = list(model.batch_generate(texts, voices=voices, instructs=instructs, lang_code="english", max_tokens=max_tokens, stream=True,
                                    streaming_interval=1e6))
    del tok.decoder.__dict__["chunked_decode"]
    calls = list(model.tokenizer.calls)
    out["batch_meta"] = json.dumps({"texts": texts, "voices": voices, "instructs": instructs, "lang_code": "english", "max_tokens": max_tokens,
                                    "tokenizer_calls": calls, "draws_left": len(mx.random.queue), "order": [int(r.sequence_idx) for r in res]})
    out["batch_u"] = ub
    for r, c in zip(res, seen):
        b = int(r.sequence_idx)
        out[f"batch_codes_{b}"] = c[0].T                              # [frames, groups]
        out[f"batch_audio_{b}"] = np.asarray(r.audio)
        print("batch row", b, "frames", c.shape[-1], "audio", r.audio.shape)
    print("batch draws left", len(mx.random.queue), "tokenizer calls", [len(c) for c in calls])
    mx.random.queue[:] = []
    session_cases(out, model, tok, texts, voices, instructs)


def session_cases(out, model, tok, texts, voices, instructs):
    """The DEFAULT batch path: Model.batch_generate(stream=False) -> Qwen3TTSBatchSession (continuous_batching.py): prompts admitted
    together with left padding, finished rows LEAVE the batch (BatchKVCache rows extracted / merged every step), each row follows the
    single-sequence trailing-text rule, and every finished row is decoded by _decode_generated_codes (15-frame chunks with 5 frames of
    left context, qwen3_tts.py:1050-1083).  Each row draws from its own uniform stream u[row, frame, group]."""
    from mlx_audio.tts.models.qwen3_tts import continuous_batching as CB
    max_tokens, g, B = 20, TALKER["num_code_groups"], len(texts)
    us = np.random.default_rng(int(os.environ.get("SEED_S", "63"))).random((B, max_tokens, g))
    state = {"rows": [], "frame": {b: 0 for b in range(B)}, "group": 0}

    def draw(shape):
        rows = state["rows"]
        assert shape == (len(rows),), (shape, rows)
        v = np.array([us[r, state["frame"][r], state["group"]] for r in rows])
        state["group"] += 1
        if state["group"] == g:
            state["group"] = 0
            for r in rows:
                state["frame"][r] += 1
        return v
    admit, advance = CB.Qwen3TTSBatchSession._admit_pending, CB.Qwen3TTSBatchSession._advance_active

    def admit_spy(self):
        state["rows"] = [it.sequence_id for it in self._pending[: min(self.available_slots, len(self._pending))]]
        return admit(self)

    def advance_spy(self):
        state["rows"] = [st.sequence_id for st in self._active]
        return advance(self)
    CB.Qwen3TTSBatchSession._admit_pending, CB.Qwen3TTSBatchSession._advance_active = admit_spy, advance_spy
    decoded = []
    real = model._decode_generated_codes

    def decode_spy(codes, **k):
        decoded.append(np.concatenate([np.asarray(c) for c in codes], axis=0))
        return real(codes, **k)
    model._decode_generated_codes = decode_spy
    mx.random.queue[:] = [("categorical", draw)] * (max_tokens * g + g)
    model.tokenizer.calls.clear()
    res = list(model.batch_generate(texts, voices=voices, instructs=instructs, lang_code="english", max_tokens=max_tokens, stream=False))
    CB.Qwen3TTSBatchSession._admit_pending, CB.Qwen3TTSBatchSession._advance_active = admit, advance
    del model.__dict__["_decode_generated_codes"]
    out["session_meta"] = json.dumps({"texts": texts, "voices": voices, "instructs": instructs, "lang_code": "english", "max_tokens": max_tokens,
                                      "tokenizer_calls": list(model.tokenizer.calls), "order": [int(r.sequence_idx) for r in res],
                                      "frames": [int(state["frame"][b]) for b in range(B)]})
    out["session_u"] = us
    for r, c in zip(res, decoded):
        b = int(r.sequence_idx)
        out[f"session_codes_{b}"], out[f"session_audio_{b}"] = c, np.asarray(r.audio)
        print("session row", b, "frames", c.shape, "audio", r.audio.shape, "token_count", r.token_count)
    mx.random.queue[:] = []


SPK = dict(mel_dim=128, enc_dim=64, enc_channels=[32, 32, 32, 32, 96], enc_kernel_sizes=[5, 3, 3, 3, 1], enc_dilations=[1, 2, 3, 4, 1],
           enc_attention_channels=16, enc_res2net_scale=4, enc_se_channels=16)


def speaker_cases(out):
    """ECAPA-TDNN speaker encoder on the reference's own 24 kHz mel front end (qwen3_tts.py:64-121, speaker_encoder.py)."""
    from mlx_audio.tts.models.qwen3_tts import qwen3_tts as Q
    from mlx_audio.tts.models.qwen3_tts import speaker_encoder as SE
    enc = SE.Qwen3TTSSpeakerEncoder(C.Qwen3TTSSpeakerEncoderConfig(**SPK))
    names = fill(enc, prefix="speaker_encoder.")
    out["spk_params"], out["spk_cfg"] = synth_params.manifest(names), json.dumps(SPK)
    audio = 0.3 * np.random.default_rng(135).standard_normal((2, 9000))                       # regenerated by the test from the seed
    mel = Q.mel_spectrogram(mx.array(audio))
    emb = enc(mel)
    out["spk_mel"], out["spk_embedding"] = np.asarray(mel), np.asarray(emb)
    print("speaker", np.asarray(mel).shape, np.asarray(emb).shape)
    return enc


def icl_cases(out, tok_full):
    """Voice cloning: Model.generate(text, ref_audio, ref_text) on a base model -> _generate_icl (qwen3_tts.py:2200-2510): reference audio
    through the speech-tokenizer encoder and the ECAPA speaker encoder, in-context prompt, the frame loop with repetition penalty 1.5,
    joint decode of [reference | generated] codes with the reference's share cut off."""
    from mlx_audio.tts.models.qwen3_tts import qwen3_tts as Q
    from mlx_audio.tts.models.qwen3_tts import speech_tokenizer as S
    Q.load_audio = lambda a, sample_rate=None: a
    mx.random.strict = False                                         # parameter initialisers draw while the modules are built
    enc4 = dict(TOKENC, num_quantizers=4)                            # the encoder must emit as many code books as the talker predicts
    tok = S.Qwen3TTSSpeechTokenizer(C.Qwen3TTSTokenizerConfig(decoder_config=C.Qwen3TTSTokenizerDecoderConfig(**TOKDEC),
                                                              encoder_config=C.Qwen3TTSTokenizerEncoderConfig(**enc4)))
    fill(tok, rule=lambda n: "small" if n.endswith((".alpha", ".beta")) else ("scale0.08" if n == "decoder.decoder.6.conv.weight" else None))
    cfg = C.ModelConfig(talker_config=dict(TALKER), speaker_encoder_config=dict(SPK), tts_model_type="base", tts_pad_token_id=111,
                        tts_bos_token_id=112, tts_eos_token_id=113)
    model = Q.Model(cfg)
    fill(model.talker)
    fill(model.speaker_encoder, prefix="speaker_encoder.")
    eos, gain = TALKER["codec_eos_token_id"], float(out["gen_eos_gain"])
    w = np.array(model.talker.codec_head.weight)
    w[eos] *= gain
    model.talker.codec_head.weight = mx.array(w)
    model.load_speech_tokenizer(tok)
    model.tokenizer = CharTokenizer()
    mx.random.strict = True
    for tag, seed in (("a", 46), ("b", 48)):                         # a: runs to max_tokens and contains a zero first code (shorter valid length); b: EOS
        rng = np.random.default_rng(seed)
        ref_audio = 0.3 * rng.standard_normal(3 * 1920 + 500)
        max_tokens, g = 10, TALKER["num_code_groups"]
        us = rng.random((max_tokens, g))
        model.tokenizer.calls.clear()
        model._icl_cache.clear()
        ie, tr, pad, ref_codes = model._prepare_icl_generation_inputs("Clone me.", mx.array(ref_audio), "Reference words", language="german")
        calls = list(model.tokenizer.calls)
        model._icl_cache.clear()
        mx.random.queue[:] = [("categorical", np.array([v])) for v in us.reshape(-1)]
        res = list(model.generate(text="Clone me.", ref_audio=mx.array(ref_audio), ref_text="Reference words", lang_code="german", max_tokens=max_tokens))
        out[f"icl_{tag}_meta"] = json.dumps({"text": "Clone me.", "ref_text": "Reference words", "lang_code": "german", "max_tokens": max_tokens,
                                             "ref_ids": calls[0], "target_ids": calls[1], "draws_left": len(mx.random.queue), "enc_nq": 4,
                                             "repetition_penalty": 1.5, "token_count": int(res[0].token_count), "seed": seed})
        out[f"icl_{tag}_ref_codes"] = np.asarray(ref_codes)            # ref_audio and u: default_rng(seed) replayed by the test
        out[f"icl_{tag}_input_embeds"], out[f"icl_{tag}_audio"] = np.asarray(ie), np.asarray(res[0].audio)
        out[f"icl_{tag}_speaker_embed"] = np.asarray(model.extract_speaker_embedding(mx.array(ref_audio)))
        print("icl", tag, "ref codes", np.asarray(ref_codes).shape, "prompt", np.asarray(ie).shape, "audio", res[0].audio.shape, "tokens", res[0].token_count,
              "draws left", len(mx.random.queue))
    mx.random.queue[:] = []
    mx.random.strict = False


def main():
    out = {"cfg": json.dumps(ORACLE_CFG)}
    talker_cases(out)
    speaker_cases(out)
    tok = tokenizer_cases(out)
    model_cases(out, tok)
    icl_cases(out, tok)
    for k in list(out):                                              # waveforms are stored as float32 (|x| <= 1: 6e-8 absolute)
        if k.endswith(("_wav", "_audio", "_wav_chunked")) or k.startswith(("batch_audio_", "session_audio_")):   # (inputs are named *_pcm_in and stay float64)
            out[k] = np.asarray(out[k], dtype=np.float32)
    np.savez_compressed(os.path.join(os.environ.get("GOLDEN_OUT", HERE), "qwen3_golden.npz"), **out)
    print({k: getattr(v, "shape", None) for k, v in out.items()})


def live(n):
    """--live N: N random configurations of the talker / code predictor / tokenizer decoder, reference classes vs oracle/qwen3.py."""
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import qwen3 as OQ
    from live_tape import Tape
    tape = Tape("qwen3", n, sys.argv)
    if tape.reference:
        from mlx_audio.tts.models.qwen3_tts import speech_tokenizer as S
    worst = 0.0
    for seed in range(n):
        rng = np.random.default_rng(2000 + seed)
        kv = int(rng.choice([1, 2]))
        heads = kv * int(rng.choice([1, 2, 4]))
        hd = int(rng.choice([8, 16, 32]))
        half = hd // 2
        a = int(rng.integers(1, half - 1))
        b = int(rng.integers(1, half - a))
        sec = [a, b, half - a - b]
        hidden, cph = int(rng.choice([32, 48])), int(rng.choice([24, 32]))
        g = int(rng.integers(2, 6))
        cp = dict(vocab_size=int(rng.integers(20, 60)), hidden_size=cph, intermediate_size=2 * cph, num_hidden_layers=int(rng.integers(1, 3)),
                  num_attention_heads=heads, num_key_value_heads=kv, head_dim=hd, num_code_groups=g)
        tk = dict(vocab_size=int(rng.integers(1100, 1200)), hidden_size=hidden, intermediate_size=2 * hidden, num_hidden_layers=int(rng.integers(1, 4)),
                  num_attention_heads=heads, num_key_value_heads=kv, head_dim=hd,
                  rope_scaling={"interleaved": True, "mrope_section": sec, "rope_type": "default"}, num_code_groups=g, text_hidden_size=24,
                  text_vocab_size=40, code_predictor_config=cp)
        oc = {"vocab_size": tk["vocab_size"], "hidden_size": hidden, "intermediate_size": 2 * hidden, "num_hidden_layers": tk["num_hidden_layers"],
              "num_attention_heads": heads, "num_key_value_heads": kv, "head_dim": hd, "rms_norm_eps": 1e-6, "rope_theta": 1000000.0,
              "mrope_section": sec, "num_code_groups": g, "codec_eos_token_id": 2150, "text_hidden_size": 24, "cp_vocab_size": cp["vocab_size"],
              "cp_hidden_size": cph, "cp_intermediate_size": 2 * cph, "cp_num_hidden_layers": cp["num_hidden_layers"], "cp_num_attention_heads": heads,
              "cp_num_key_value_heads": kv, "cp_head_dim": hd, "cp_rope_theta": 1000000.0}
        if tape.reference:
            talker = T.Qwen3TTSTalkerForConditionalGeneration(C.Qwen3TTSTalkerConfig(**tk))
        P = {k: torch.as_tensor(synth_params.value(k, sh, r)) for k, sh, r in tape.value(lambda: fill(talker))}
        bsz, s0 = int(rng.integers(1, 4)), int(rng.integers(2, 9))
        x = rng.standard_normal((bsz, s0, hidden))
        ocache = OQ.make_cache(oc["num_hidden_layers"])
        if tape.reference:
            cache = talker.make_cache()
            lg, _ = talker(mx.array(x), cache=cache)
        olg, _ = OQ.talker_forward(P, torch.as_tensor(x), ocache, cfg=oc)
        errs = [tape.err(lambda: lg, olg.numpy())]
        for _ in range(2):
            x1 = rng.standard_normal((bsz, 1, hidden))
            if tape.reference:
                lg, _ = talker(mx.array(x1), cache=cache)
            olg, _ = OQ.talker_forward(P, torch.as_tensor(x1), ocache, cfg=oc)
            errs.append(tape.err(lambda: lg, olg.numpy()))
        occ = OQ.make_cache(oc["cp_num_hidden_layers"])
        if tape.reference:
            cc = talker.code_predictor.make_cache()
        cx = rng.standard_normal((bsz, 2, hidden))
        if tape.reference:
            cl, cc, _ = talker.code_predictor(mx.array(cx), cache=cc, generation_step=0)
        errs.append(tape.err(lambda: cl, OQ.code_predictor_forward(P, torch.as_tensor(cx), occ, 0, oc).numpy()))
        for st in range(1, g - 1):
            c1 = rng.standard_normal((bsz, 1, hidden))
            if tape.reference:
                cl, cc, _ = talker.code_predictor(mx.array(c1), cache=cc, generation_step=st)
            errs.append(tape.err(lambda: cl, OQ.code_predictor_forward(P, torch.as_tensor(c1), occ, st, oc).numpy()))
        # tokenizer decoder with other strides
        ups = [int(v) for v in rng.choice([2, 3, 4, 5], size=int(rng.integers(2, 4)))]
        rat = [int(v) for v in rng.choice([2, 3], size=int(rng.integers(1, 3)))]
        dh = int(rng.choice([1, 2, 4]))
        dd = 8 * 2 ** len(ups)
        nq = int(rng.integers(2, 6))
        td = dict(latent_dim=24, codebook_dim=8, codebook_size=32, decoder_dim=dd, hidden_size=dh * 8, intermediate_size=32, head_dim=8,
                  num_attention_heads=dh, num_hidden_layers=int(rng.integers(1, 3)), num_key_value_heads=dh, num_quantizers=nq,
                  num_semantic_quantizers=1, upsample_rates=ups, upsampling_ratios=rat)
        otd = {"latent_dim": 24, "codebook_dim": 8, "codebook_size": 32, "decoder_dim": dd, "hidden_size": dh * 8, "intermediate_size": 32,
               "layer_scale_initial_scale": 0.01, "head_dim": 8, "num_attention_heads": dh, "num_hidden_layers": td["num_hidden_layers"],
               "num_key_value_heads": dh, "num_quantizers": nq, "num_semantic_quantizers": 1, "rms_norm_eps": 1e-5, "rope_theta": 10000.0,
               "upsample_rates": ups, "upsampling_ratios": rat}
        if tape.reference:
            tok = S.Qwen3TTSSpeechTokenizer(C.Qwen3TTSTokenizerConfig(decoder_config=C.Qwen3TTSTokenizerDecoderConfig(**td)))
        names = tape.value(lambda: fill(tok, rule=lambda nm: "small" if nm.endswith((".alpha", ".beta")) else None))
        PT = {k: torch.as_tensor(synth_params.value(k, sh, r)) for k, sh, r in names}
        codes = rng.integers(0, 32, size=(2, nq, int(rng.integers(2, 7))))
        if tape.reference:
            wav = np.asarray(tok.decoder(mx.array(codes)))
        owav = OQ.tokenizer_decode(PT, torch.as_tensor(codes), otd).numpy()
        errs.append(tape.err(lambda: wav, owav))
        worst = max(worst, float(max(errs)))
        print("qwen3 heads", heads, "kv", kv, "hd", hd, "mrope", sec, "groups", g, "| tokenizer ups", ups, rat, "nq", nq, "max err", float(max(errs)))
    # sampler chain (qwen3_tts.py:805-860 over lm/sample_utils.py): random logits and settings, the same injected uniform on both sides
    if tape.reference:
        from mlx_audio.tts.models.qwen3_tts import qwen3_tts as QM
        m = QM.Model.__new__(QM.Model)
        mx.random.strict = True
    n_cases = 60 * n
    for case in range(n_cases):
        rng = np.random.default_rng(9000 + case)
        V = int(rng.integers(8, 300))
        logits = rng.standard_normal(V) * float(rng.choice([0.5, 2.0, 6.0]))
        kw = dict(temperature=float(rng.choice([0.0, 0.3, 0.9, 1.0, 1.7])), top_k=int(rng.choice([0, 1, 5, 50, 400])),
                  top_p=float(rng.choice([1.0, 0.95, 0.7, 0.2])), repetition_penalty=float(rng.choice([1.0, 1.05, 1.5])),
                  min_p=float(rng.choice([0.0, 0.0, 0.05, 0.3])))
        gen = [int(v) for v in rng.integers(0, V + 20, size=int(rng.integers(0, 8)))] or None
        sup = [int(v) for v in rng.choice(V, size=int(rng.integers(0, max(1, V // 4))), replace=False)] or None
        if sup is not None and len(sup) >= V:
            sup = sup[: V - 1]
        u = float(rng.random())

        def ref_token():
            mx.random.queue[:] = [("categorical", np.array([u]))]
            t = int(np.asarray(m._sample_token(mx.array(logits[None, None, :]), generated_tokens=gen, suppress_tokens=sup, **kw))[0, 0])
            mx.random.queue[:] = []
            return t
        tok = tape.value(ref_token)
        want = OQ.sample_token(torch.as_tensor(logits), u, kw["temperature"], kw["top_k"], kw["top_p"], kw["repetition_penalty"], gen, sup, kw["min_p"])
        assert tok == want, (case, kw, tok, want)
    mx.random.strict = False
    tape.close()
    print("sampler cases identical:", n_cases)
    assert worst < 1e-9, worst
    print("LIVE OK", worst)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--live":
        live(int(sys.argv[2]))
    else:
        main()
