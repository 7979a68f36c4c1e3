"""Golden vectors from the REFERENCE'S OWN Kokoro code (tts/models/kokoro/{kokoro,modules,istftnet}.py, tts/models/interpolate.py,
dsp.py) executed in float64 with NumPy standing in for MLX (numpy_mlx_nn.py), on the public Kokoro-82M configuration with the
synthetic weights of mlx_audio_b200/synth.py (the same weights the GPU parity tests use).  Run from the repo root in the build
container:  python tests/golden/make_kokoro_golden.py  ->  tests/golden/kokoro_golden.npz

The two MLX random draws of the source module (initial harmonic phases, additive noise; istftnet.py:581,649) are injected."""
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
import numpy_mlx_nn as shim          # noqa: E402

REF = "/root/reference/mlx_audio"
mx, nn = shim.install(precise=True)
if "--replay" not in sys.argv:                                 # replaying a --live record needs no reference source
    for name, path in (("mlx_audio", REF), ("mlx_audio.tts", f"{REF}/tts"), ("mlx_audio.tts.models", f"{REF}/tts/models"),
                       ("mlx_audio.tts.models.kokoro", f"{REF}/tts/models/kokoro")):
        shim.stub_package(name, path)
    hub = types.ModuleType("huggingface_hub")
    hub.snapshot_download = hub.hf_hub_download = None
    sys.modules["huggingface_hub"] = hub
    import mlx_audio.dsp as _dsp          # noqa: E402
    u = types.ModuleType("mlx_audio.utils")
    u.load_audio = None
    for n in ("hanning", "mel_filters", "stft", "istft"):
        setattr(u, n, getattr(_dsp, n))
    sys.modules["mlx_audio.utils"] = u
    from mlx_audio.tts.models.kokoro import kokoro as K          # noqa: E402

# The harmonic source's STFT phase (istftnet.py:473-505: arctan2(imag, real)) is ill-defined wherever a bin is exactly real -- DC,
# Nyquist, and every bin of the reflect-symmetric first frame: there the imaginary part is FFT rounding noise (or a signed zero)
# and its sign picks +pi or -pi, in MLX's FFT as in NumPy's.  The oracle and the CUDA kernel canonicalise such bins to +0
# (oracle/kokoro.py:mlxstft_transform); the stand-in FFT does the same so that the run is deterministic on this point.
_rfft = mx.fft.rfft


def _rfft_canonical(x, n=None, axis=-1, **k):
    y = np.asarray(_rfft(x, n=n, axis=axis, **k))
    im = np.where(np.abs(y.imag) <= 1e-12 * np.abs(y.real), 0.0, y.imag)
    return (y.real + 1j * im).view(shim.array)


mx.fft.rfft = _rfft_canonical

sys.path.insert(0, ROOT)
import importlib.util                 # noqa: E402
spec = importlib.util.spec_from_file_location("b200_synth", os.path.join(ROOT, "mlx_audio_b200", "synth.py"))
synth = importlib.util.module_from_spec(spec)
spec.loader.exec_module(synth)
from oracle.kokoro import KOKORO_CONFIG                      # noqa: E402  (a dict of constants, the public config)


def main():
    cfg = json.loads(json.dumps(KOKORO_CONFIG))
    vocab = {chr(0x100 + i): i for i in range(cfg["n_token"])}
    model = K.Model(K.ModelConfig(**cfg, vocab=vocab))
    model.eval()
    P = synth.kokoro_weights(cfg, seed=0)
    have = dict(shim.flat_parameters(model))
    missing, extra = sorted(set(have) - set(P)), sorted(set(P) - set(have))
    print("reference parameters", len(have), "synthetic", len(P), "missing", missing[:5], "extra", extra[:5])
    assert not missing and not extra
    f0_gain = 600.0                                                  # synthetic F0 is ~+-0.3; scaled into +-200 Hz so that voiced frames exist
    P["predictor.F0_proj.weight"] = P["predictor.F0_proj.weight"] * f0_gain
    for n, v in P.items():
        assert tuple(have[n].shape) == tuple(v.shape), (n, have[n].shape, v.shape)
        shim.set_parameter(model, n, v.double().numpy())
    n_ph = int(os.environ.get("N_PH", "10"))
    ids, ref_s = synth.kokoro_inputs(n_ph, cfg["n_token"], seed=1)
    ids = np.asarray(ids)[0]
    phonemes = "".join(chr(0x100 + int(i)) for i in ids[1:-1])
    rng = np.random.default_rng(71)
    rand_ini = rng.random((1, 9))
    draws = {}

    def noise(shape):
        draws["noise"] = rng.standard_normal(shape).astype(np.float32).astype(np.float64)      # stored as float32, exactly
        return draws["noise"]
    mx.random.strict = True
    mx.random.queue[:] = [("uniform", rand_ini), ("normal", noise), ("normal", lambda shape: np.zeros(shape))]
    res = model(phonemes, mx.array(np.asarray(ref_s, dtype=np.float64)), speed=float(os.environ.get("SPEED", "0.5")), return_output=True)
    assert not mx.random.queue
    audio, pred_dur = np.asarray(res.audio), np.asarray(res.pred_dur)
    print("pred_dur", pred_dur.tolist(), "audio", audio.shape, float(np.abs(audio).max()))
    np.savez_compressed(os.path.join(os.environ.get("GOLDEN_OUT", HERE), "kokoro_golden.npz"), ids=ids, ref_s=np.asarray(ref_s, dtype=np.float64), rand_ini=rand_ini,
                        noise_shape=np.asarray(draws["noise"].shape), pred_dur=pred_dur, audio=audio.astype(np.float32),
                        meta=json.dumps({"n_phonemes": n_ph, "weights": "synth.kokoro_weights(KOKORO_CONFIG, seed=0)", "f0_gain": f0_gain, "noise": "np.random.default_rng(71): .random((1, 9)) then .standard_normal(noise_shape).astype(float32)", "speed": float(os.environ.get("SPEED", "0.5"))}))


def live(n):
    """--live N: N random utterances (length, speed, style vector, weight seed, F0 scale) through the reference Model.__call__ and the
    oracle's forward; durations identical, waveform 1e-9."""
    import torch
    from oracle import kokoro as OK
    from live_tape import Tape
    tape = Tape("kokoro", n, sys.argv)
    OK.EFFECTIVE_WEIGHTS_BF16 = False
    cfg = json.loads(json.dumps(KOKORO_CONFIG))
    vocab = {chr(0x100 + i): i for i in range(cfg["n_token"])}
    if tape.reference:
        model = K.Model(K.ModelConfig(**cfg, vocab=vocab))
        model.eval()
    worst = 0.0
    for seed in range(n):
        rng = np.random.default_rng(4000 + seed)
        P = synth.kokoro_weights(cfg, seed=int(rng.integers(1, 100)))
        P["predictor.F0_proj.weight"] = P["predictor.F0_proj.weight"] * float(rng.uniform(200, 900))
        if tape.reference:
            for k, v in P.items():
                shim.set_parameter(model, k, v.double().numpy())
        n_ph, speed = int(rng.integers(3, 14)), float(rng.uniform(0.4, 1.2))
        ids = rng.integers(1, cfg["n_token"], size=n_ph)
        ref_s = rng.standard_normal((1, 256))
        rand_ini = rng.random((1, 9))
        draws = {}

        def noise(shape):
            draws["noise"] = rng.standard_normal(shape)
            return draws["noise"]
        if tape.reference:
            mx.random.strict = True
            mx.random.queue[:] = [("uniform", rand_ini), ("normal", noise), ("normal", lambda shape: np.zeros(shape))]
            res = model("".join(chr(0x100 + int(i)) for i in ids), mx.array(ref_s), speed=speed, return_output=True)
            mx.random.strict = False
        shape = tape.value(lambda: draws["noise"].shape)
        if not tape.reference:
            noise(shape)                                       # the draw the reference's call made, from the same generator state
        audio, pd = OK.forward({k: v.double() for k, v in P.items()}, torch.as_tensor(np.concatenate([[0], ids, [0]]))[None], torch.as_tensor(ref_s), cfg,
                               speed=speed, rand_ini=torch.as_tensor(rand_ini), noise=torch.as_tensor(draws["noise"]))
        pred_dur = tape.value(lambda: np.asarray(res.pred_dur))
        assert np.array_equal(pd.numpy(), np.asarray(pred_dur)), (pd, pred_dur)
        err = tape.err(lambda: np.asarray(res.audio).reshape(-1), audio.numpy().reshape(-1), sample=512)
        worst = max(worst, err)
        print("kokoro phonemes", n_ph, "speed", round(speed, 2), "durations", pred_dur, "samples", audio.numel(), "err", err)
    tape.close()
    assert worst < 2e-8, worst          # float64 on both sides; the harmonic phase integrates over every frame, so the error grows with the
                                        # utterance (measured: 1.4e-9 at 58 frames, 3-6 frames per phoneme)
    print("LIVE OK", worst)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--live":
        live(int(sys.argv[2]))
    else:
        main()
