"""Golden vectors from the REFERENCE'S OWN codec code (codec/models/snac/*.py, codec/models/mimi/**) executed in float64 with
NumPy standing in for MLX (numpy_mlx_nn.py), at reduced configurations.  Run from the repo root in the build container:
python tests/golden/make_codec_golden.py  ->  tests/golden/codec_golden.npz"""
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
    for name, path in (("mlx_audio", REF), ("mlx_audio.lm", f"{REF}/lm"), ("mlx_audio.lm.models", f"{REF}/lm/models"), ("mlx_audio.codec", f"{REF}/codec"),
                       ("mlx_audio.codec.models", f"{REF}/codec/models"), ("mlx_audio.codec.models.snac", f"{REF}/codec/models/snac"),
                       ("mlx_audio.codec.models.mimi", f"{REF}/codec/models/mimi")):
        shim.stub_package(name, path)
hub = types.ModuleType("huggingface_hub")
hub.snapshot_download = hub.hf_hub_download = None
sys.modules["huggingface_hub"] = hub

SNAC_CFG = dict(sampling_rate=24000, encoder_dim=8, encoder_rates=[2, 2, 2, 2], latent_dim=None, decoder_dim=64, decoder_rates=[8, 3, 4, 2],
                attn_window_size=None, codebook_size=64, codebook_dim=4, vq_strides=[4, 2, 1], noise=True, depthwise=True)


def fill(module, prefix="", rule=lambda name: None):
    names = [(prefix + n, v.shape, rule(n)) for n, v in shim.flat_parameters(module)]
    for n, sh, r in names:
        shim.set_parameter(module, n[len(prefix):], synth_params.value(n, sh, r))
    for m in module.modules():                                       # derived buffers (Mimi codebooks: embedding_sum / usage), as the
        if hasattr(m, "update_in_place"):                            # reference's own weight loader does after assigning parameters
            m.update_in_place()
    return names


def snac_cases(out):
    from mlx_audio.codec.models.snac import snac as S
    model = S.SNAC(**SNAC_CFG)
    import re
    last = max(int(m.group(1)) for n, _ in shim.flat_parameters(model) if (m := re.match(r"decoder\.model\.layers\.(\d+)\.weight_g$", n)))
    names = fill(model, rule=lambda n: "scale0.03" if n == f"decoder.model.layers.{last}.weight_g" else None)   # keeps tanh mostly unsaturated
    out["snac_params"], out["snac_cfg"] = synth_params.manifest(names), json.dumps(SNAC_CFG)
    rng = np.random.default_rng(61)
    t = 5
    codes = [rng.integers(0, 64, size=(2, t * 4 // s)) for s in SNAC_CFG["vq_strides"]]
    chans = [SNAC_CFG["decoder_dim"] // 2 ** (i + 1) for i in range(4)]
    noises = [rng.standard_normal((2, 1, c)) for c in chans]
    mx.random.strict = True
    mx.random.queue[:] = [("normal", n) for n in noises]
    audio = model.decode([mx.array(c) for c in codes])
    assert not mx.random.queue
    mx.random.strict = False
    # encode side: audio -> three code streams (integer result); 700 samples short of the padding quantum
    audio_in = 0.5 * rng.standard_normal((2, 1, 3 * 64 - 50))
    enc = model.encode(mx.array(audio_in))
    out["snac_enc_audio"] = audio_in
    for i, c in enumerate(enc):
        out[f"snac_enc_codes_{i}"] = np.asarray(c)
    print("snac encode", [np.asarray(c).shape for c in enc])
    # decode_stream: a first call and a second call that prepends context (two decodes = eight noise draws)
    c1 = [rng.integers(0, 64, size=(2, 12 // s_)) for s_ in SNAC_CFG["vq_strides"]]
    c2 = [rng.integers(0, 64, size=(2, 8 // s_)) for s_ in SNAC_CFG["vq_strides"]]
    zs = [rng.standard_normal((2, 1, c)) for c in chans] + [rng.standard_normal((2, 1, c)) for c in chans]
    mx.random.strict = True
    mx.random.queue[:] = [("normal", z) for z in zs]
    a1, ctx = model.decode_stream([mx.array(c) for c in c1])
    a2, ctx2 = model.decode_stream([mx.array(c) for c in c2], prev_codes=ctx, context_frames=8)
    assert not mx.random.queue
    mx.random.strict = False
    for i in range(3):
        out[f"snac_stream_c1_{i}"], out[f"snac_stream_c2_{i}"], out[f"snac_stream_ctx_{i}"] = c1[i], c2[i], np.asarray(ctx2[i])
    for i, z in enumerate(zs):
        out[f"snac_stream_noise_{i}"] = z
    out["snac_stream_audio1"], out["snac_stream_audio2"] = np.asarray(a1), np.asarray(a2)
    print("snac decode_stream", np.asarray(a1).shape, np.asarray(a2).shape, [np.asarray(c).shape for c in ctx2])
    for i, c in enumerate(codes):
        out[f"snac_codes_{i}"] = c
    for i, n in enumerate(noises):
        out[f"snac_noise_{i}"] = n
    out["snac_audio"] = np.asarray(audio)
    print("snac audio", audio.shape, "saturated", float((np.abs(np.asarray(audio)) > 0.999).mean()))


MIMI_ORACLE = {"dimension": 32, "nfilters": 4, "ratios": [8, 6, 5, 4], "ksize": 7, "residual_ksize": 3, "last_ksize": 3, "compress": 2, "d_model": 32,
               "num_heads": 4, "num_layers": 2, "dim_feedforward": 64, "context": 6, "max_period": 10000, "layer_scale": 0.01, "nq": 4, "bins": 64,
               "qdim": 16, "upsample_stride": 2}


def mimi_cases(out):
    from mlx_audio.codec.models.mimi import mimi as M
    from mlx_audio.codec.models.mimi.modules import SeanetConfig, TransformerConfig
    c = MIMI_ORACLE
    seanet = SeanetConfig(dimension=c["dimension"], channels=1, causal=True, nfilters=c["nfilters"], nresidual_layers=1, ratios=c["ratios"],
                          ksize=c["ksize"], residual_ksize=c["residual_ksize"], last_ksize=c["last_ksize"], dilation_base=2, pad_mode="constant",
                          true_skip=True, compress=c["compress"])
    tr = TransformerConfig(d_model=c["d_model"], num_heads=c["num_heads"], num_layers=c["num_layers"], causal=True, norm_first=True, bias_ff=False,
                           bias_attn=False, layer_scale=c["layer_scale"], positional_embedding="rope", use_conv_bias=True, gating=False,
                           norm="layer_norm", context=c["context"], max_period=c["max_period"], max_seq_len=8192, kv_repeat=1,
                           dim_feedforward=c["dim_feedforward"], conv_layout=True, use_conv_block=False, cross_attention=False, conv_kernel_size=3)
    cfg = M.MimiConfig(channels=1, sample_rate=24000, frame_rate=12.5, renormalize=True, seanet=seanet, transformer=tr, quantizer_nq=c["nq"],
                       quantizer_bins=c["bins"], quantizer_dim=c["qdim"])
    model = M.Mimi(cfg)
    names = fill(model)
    out["mimi_params"], out["mimi_cfg"] = synth_params.manifest(names), json.dumps(c)
    rng = np.random.default_rng(62)
    codes = rng.integers(0, c["bins"], size=(2, c["nq"], 9))
    pcm = model.decode(mx.array(codes))
    out["mimi_codes"], out["mimi_pcm"] = codes, np.asarray(pcm)
    print("mimi pcm", pcm.shape, float(np.abs(np.asarray(pcm)).max()))
    # encode side: pcm -> codes (integer result), an input length that is not a multiple of the 1920-sample frame
    pcm_in = 0.5 * rng.standard_normal((2, 1, 12 * 1920 + 700))
    out["mimi_enc_pcm"], out["mimi_enc_codes"] = pcm_in, np.asarray(model.encode(mx.array(pcm_in)))
    print("mimi encode", out["mimi_enc_codes"].shape)
    # streaming: decode_step over two chunks continues the conv buffers and the rotating kv cache
    model.reset_state()
    parts = [np.asarray(model.decode_step(mx.array(codes[:, :, :4]))), np.asarray(model.decode_step(mx.array(codes[:, :, 4:])))]
    out["mimi_pcm_steps"] = np.concatenate(parts, axis=-1)
    print("mimi step vs full", float(np.abs(out["mimi_pcm_steps"] - out["mimi_pcm"]).max()))


def main():
    out = {}
    snac_cases(out)
    mimi_cases(out)
    out.pop("mimi_pcm_steps")                                        # equal to the one-shot decode (checked above)
    for k in ("snac_audio", "mimi_pcm", "snac_stream_audio1", "snac_stream_audio2"):                             # waveforms stored as float32 (|x| <= 1: 6e-8 absolute)
        out[k] = np.asarray(out[k], dtype=np.float32)
    np.savez_compressed(os.path.join(os.environ.get("GOLDEN_OUT", HERE), "codec_golden.npz"), **out)
    print({k: getattr(v, "shape", None) for k, v in out.items()})


def live(n):
    """--live N: N random SNAC / Mimi configurations, the reference's encode and decode vs oracle/codec.py (codes must be identical)."""
    import re
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import codec as OC
    from live_tape import Tape
    tape = Tape("codec", n, sys.argv)
    if tape.reference:
        from mlx_audio.codec.models.mimi import mimi as M
        from mlx_audio.codec.models.mimi.modules import SeanetConfig, TransformerConfig
        from mlx_audio.codec.models.snac import snac as S
    worst = 0.0
    for seed in range(n):
        rng = np.random.default_rng(3000 + seed)
        nr = int(rng.integers(2, 5))
        drates = [int(v) for v in rng.choice([2, 3, 4, 5, 8], size=nr)]
        erates = [int(v) for v in rng.choice([2, 3, 4], size=int(rng.integers(2, 4)))]
        vs = [[4, 2, 1], [2, 1], [1, 1], [8, 4, 2, 1]][int(rng.integers(0, 4))]
        cfg = dict(sampling_rate=24000, encoder_dim=int(rng.choice([4, 8])), encoder_rates=erates, latent_dim=None, decoder_dim=8 * 2 ** nr,
                   decoder_rates=drates, attn_window_size=None, codebook_size=int(rng.integers(16, 64)), codebook_dim=int(rng.choice([4, 8])),
                   vq_strides=vs, noise=bool(rng.integers(0, 2)), depthwise=bool(rng.integers(0, 2)))
        if tape.reference:
            model = S.SNAC(**cfg)
            last = max(int(m.group(1)) for k, _ in shim.flat_parameters(model) if (m := re.match(r"decoder\.model\.layers\.(\d+)\.weight_g$", k)))
        names = tape.value(lambda: fill(model, rule=lambda k: "scale0.03" if k == f"decoder.model.layers.{last}.weight_g" else None))
        P = {k: torch.as_tensor(synth_params.value(k, sh, r)) for k, sh, r in names}
        t = int(rng.integers(1, 4)) * vs[0]
        codes = [rng.integers(0, cfg["codebook_size"], size=(2, t // st)) for st in vs]
        noises = [rng.standard_normal((2, 1, cfg["decoder_dim"] // 2 ** (i + 1))) for i in range(nr)]
        if tape.reference:
            mx.random.strict = True
            mx.random.queue[:] = [("normal", z) for z in noises] if cfg["noise"] else []
            audio = np.asarray(model.decode([mx.array(c) for c in codes]))
            mx.random.queue[:] = []
            mx.random.strict = False
        o = OC.snac_decode(P, [torch.as_tensor(c).long() for c in codes], cfg, [torch.as_tensor(z) for z in noises]).numpy()
        errs = [tape.err(lambda: audio, o)]
        a_in = 0.5 * rng.standard_normal((2, 1, int(rng.integers(40, 400))))
        enc = tape.value(lambda: [np.asarray(e) for e in model.encode(mx.array(a_in))])
        oenc = OC.snac_encode(P, torch.as_tensor(a_in), cfg)
        assert len(enc) == len(oenc) and all(np.array_equal(np.asarray(e), oe.numpy()) for e, oe in zip(enc, oenc)), ("snac encode", cfg)
        print("snac dec", drates, "enc", erates, "vq", vs, "noise", cfg["noise"], "depthwise", cfg["depthwise"], "samples", o.shape[1], "err", float(errs[0]))
        # Mimi
        ratios = [int(v) for v in rng.choice([2, 3, 4, 5], size=int(rng.integers(2, 5)))]
        heads = int(rng.choice([1, 2, 4]))
        c = {"dimension": 8 * heads, "nfilters": int(rng.choice([2, 4])), "ratios": ratios, "ksize": int(rng.choice([3, 7])), "residual_ksize": 3,
             "last_ksize": int(rng.choice([3, 5])), "compress": 2, "d_model": 8 * heads, "num_heads": heads, "num_layers": int(rng.integers(1, 3)),
             "dim_feedforward": 32, "context": int(rng.integers(2, 12)), "max_period": 10000, "layer_scale": 0.01, "nq": int(rng.integers(1, 6)),
             "bins": int(rng.integers(8, 40)), "qdim": int(rng.choice([4, 8])), "upsample_stride": 2}
        hop = int(np.prod(ratios))
        if tape.reference:
            seanet = SeanetConfig(dimension=c["dimension"], channels=1, causal=True, nfilters=c["nfilters"], nresidual_layers=1, ratios=c["ratios"],
                                  ksize=c["ksize"], residual_ksize=c["residual_ksize"], last_ksize=c["last_ksize"], dilation_base=2, pad_mode="constant",
                                  true_skip=True, compress=c["compress"])
            tr = TransformerConfig(d_model=c["d_model"], num_heads=c["num_heads"], num_layers=c["num_layers"], causal=True, norm_first=True, bias_ff=False,
                                   bias_attn=False, layer_scale=c["layer_scale"], positional_embedding="rope", use_conv_bias=True, gating=False,
                                   norm="layer_norm", context=c["context"], max_period=c["max_period"], max_seq_len=8192, kv_repeat=1,
                                   dim_feedforward=c["dim_feedforward"], conv_layout=True, use_conv_block=False, cross_attention=False, conv_kernel_size=3)
            mm = M.Mimi(M.MimiConfig(channels=1, sample_rate=float(2 * hop * 12.5), frame_rate=12.5, renormalize=True, seanet=seanet, transformer=tr,
                                     quantizer_nq=c["nq"], quantizer_bins=c["bins"], quantizer_dim=c["qdim"]))
        P = {k: torch.as_tensor(synth_params.value(k, sh, r)) for k, sh, r in tape.value(lambda: fill(mm))}
        mc = rng.integers(0, c["bins"], size=(2, c["nq"], int(rng.integers(1, 8))))
        if tape.reference:
            pcm = np.asarray(mm.decode(mx.array(mc)))
        opcm = OC.mimi_decode(P, torch.as_tensor(mc).long(), c).numpy()
        errs.append(tape.err(lambda: pcm, opcm))
        p_in = 0.5 * rng.standard_normal((2, 1, int(rng.integers(1, 5)) * 2 * hop + int(rng.integers(0, hop))))
        assert np.array_equal(np.asarray(tape.value(lambda: np.asarray(mm.encode(mx.array(p_in))))), OC.mimi_encode(P, torch.as_tensor(p_in), c).numpy()), ("mimi encode", c)
        print("mimi ratios", ratios, "heads", heads, "context", c["context"], "nq", c["nq"], "ksize", c["ksize"], c["last_ksize"], "err", float(errs[-1]))
        worst = max(worst, float(max(errs)))
    tape.close()
    assert worst < 1e-9, worst
    print("LIVE OK", worst)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--live":
        live(int(sys.argv[2]))
    else:
        main()
