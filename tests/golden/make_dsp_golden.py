#!/usr/bin/env python
"""Golden vectors for the DSP front end produced by the REFERENCE'S OWN code (mlx_audio/dsp.py and
stt/models/whisper/audio.py:log_mel_spectrogram), executed in the build container with NumPy standing in for the MLX primitives it
calls (tests/golden/numpy_mlx_shim.py: MLX itself has no wheel here).  What is pinned is therefore the reference's control flow,
constants, padding / framing / normalisation rules -- the parts a restatement can get wrong -- on top of NumPy's definition of the
primitives.  /root/reference does not exist on the GPU box: the vectors are committed.

    python tests/golden/make_dsp_golden.py          # needs /root/reference
"""
import importlib.util
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import numpy_mlx_shim  # noqa: E402

REF = "/root/reference/mlx_audio"


def load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    spec.loader.exec_module(m)
    return m


def main():
    numpy_mlx_shim.install()
    dsp = load(os.path.join(REF, "dsp.py"), "ref_dsp")
    # stubs for audio.py's package imports: `mlx_audio.utils` re-exports dsp (utils.py:31-40), `mlx_audio.stt.utils.load_audio` is unused
    pkg = types.ModuleType("mlx_audio"); pkg.__path__ = []
    stt = types.ModuleType("mlx_audio.stt"); stt.__path__ = []
    stt_utils = types.ModuleType("mlx_audio.stt.utils"); stt_utils.load_audio = lambda *_a, **_k: (_ for _ in ()).throw(RuntimeError("no files"))
    utils = types.ModuleType("mlx_audio.utils")
    for n in ("hanning", "mel_filters", "stft"):
        setattr(utils, n, getattr(dsp, n))
    sys.modules.update({"mlx_audio": pkg, "mlx_audio.stt": stt, "mlx_audio.stt.utils": stt_utils, "mlx_audio.utils": utils})
    audio = load(os.path.join(REF, "stt/models/whisper/audio.py"), "ref_whisper_audio")

    out = {}
    for name in ("hanning", "hamming", "blackman", "bartlett"):
        for size in (20, 400):
            out[f"win_{name}_{size}"] = np.asarray(getattr(dsp, name)(size), dtype=np.float32)
            out[f"win_{name}_{size}_periodic"] = np.asarray(getattr(dsp, name)(size, periodic=True), dtype=np.float32)
    rng = np.random.default_rng(0)
    x = rng.standard_normal(4000).astype(np.float32)
    for tag, kw in (("whisper", dict(n_fft=400, hop_length=160, window="hann")), ("kokoro", dict(n_fft=20, hop_length=5, window="hann")),
                    ("const", dict(n_fft=256, hop_length=64, window="hamming", pad_mode="constant")), ("nocenter", dict(n_fft=128, hop_length=32, center=False)),
                    ("shortwin", dict(n_fft=512, hop_length=128, win_length=400))):
        s = dsp.stft(numpy_mlx_shim.array(x), **kw)
        out[f"stft_{tag}_re"], out[f"stft_{tag}_im"] = np.real(s).astype(np.float32), np.imag(s).astype(np.float32)
    s = dsp.stft(numpy_mlx_shim.array(x), n_fft=256, hop_length=64)
    # win_length is passed explicitly: the default reads the FRAME count ((x.shape[1] - 1) * 2, dsp.py:465-466), a reference quirk
    # that only works when frames == n_fft / 2 + 1 (kept in the oracle and the product, pinned in tests/test_oracle_pins.py)
    for tag, kw in (("default", dict(hop_length=64, win_length=256)), ("len", dict(hop_length=64, win_length=256, length=3900)),
                    ("norm", dict(hop_length=64, win_length=256, normalized=True))):
        out[f"istft_{tag}"] = np.asarray(dsp.istft(numpy_mlx_shim.array(np.asarray(s).T), **kw), dtype=np.float32)
    for tag, kw in (("whisper80", dict(sample_rate=16000, n_fft=400, n_mels=80, norm="slaney", mel_scale=None)),
                    ("whisper128", dict(sample_rate=16000, n_fft=400, n_mels=128, norm="slaney", mel_scale=None)),
                    ("qwen3", dict(sample_rate=24000, n_fft=1024, n_mels=128, f_min=0.0, f_max=12000.0, norm="slaney", mel_scale="slaney")),
                    ("htk", dict(sample_rate=22050, n_fft=512, n_mels=40, norm=None, mel_scale="htk"))):
        out[f"mel_{tag}"] = np.asarray(dsp.mel_filters(**kw), dtype=np.float32)
    a = (0.1 * rng.standard_normal(16000)).astype(np.float32)
    out["logmel_noise"] = np.asarray(audio.log_mel_spectrogram(a, n_mels=80, padding=0), dtype=np.float32)
    out["logmel_noise_padded"] = np.asarray(audio.log_mel_spectrogram(a[:4000], n_mels=80, padding=8000), dtype=np.float32)
    sine = np.sin(2 * np.pi * 440.0 * np.arange(16000) / 16000.0).astype(np.float32)          # BASELINE config 1
    out["logmel_sine440"] = np.asarray(audio.log_mel_spectrogram(sine, n_mels=80, padding=0), dtype=np.float32)
    np.savez_compressed(os.path.join(os.environ.get("GOLDEN_OUT", HERE), "dsp_golden.npz"), **out)
    print({k: v.shape for k, v in out.items()})


def live(n):
    """--live N: random STFT / iSTFT / mel-filterbank / log-mel configurations, the reference's dsp.py (float32, NumPy standing in for MLX)
    vs oracle/dsp.py side by side (--record / --replay: live_tape.py)."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import dsp as O
    from live_tape import Tape
    tape = Tape("dsp", n, sys.argv)
    numpy_mlx_shim.install()
    if tape.reference:
        dsp = load(os.path.join(REF, "dsp.py"), "ref_dsp_live")
    worst = {"stft": 0.0, "istft": 0.0, "mel": 0.0, "window": 0.0}
    for seed in range(n):
        rng = np.random.default_rng(5000 + seed)
        n_fft = int(rng.choice([16, 20, 64, 128, 400, 512]))
        hop = int(rng.integers(max(1, n_fft // 8), n_fft // 2 + 1))
        win_length = int(rng.choice([n_fft, max(4, n_fft - int(rng.integers(0, n_fft // 2)))]))
        window = str(rng.choice(["hann", "hamming", "blackman", "bartlett"]))
        center = bool(rng.integers(0, 2))
        pad_mode = str(rng.choice(["reflect", "constant"]))
        x = rng.standard_normal(int(rng.integers(2 * n_fft, 6 * n_fft))).astype(np.float32)
        kw = dict(n_fft=n_fft, hop_length=hop, win_length=win_length, window=window, center=center, pad_mode=pad_mode)
        b = O.stft(x, **kw)
        worst["stft"] = max(worst["stft"], tape.err(lambda: dsp.stft(numpy_mlx_shim.array(x), **kw), b) / max(1.0, np.abs(b).max()))
        for size in (int(rng.integers(3, 40)),):
            for name in ("hanning", "hamming", "blackman", "bartlett"):
                for periodic in (False, True):
                    wb = getattr(O, name)(size, periodic=periodic)
                    worst["window"] = max(worst["window"], tape.err(lambda: getattr(dsp, name)(size, periodic=periodic), wb))
        # iSTFT of a centred reflect STFT with a full-length window (the combination the reference's own callers use)
        nf = int(rng.choice([16, 64, 256]))
        hp = nf // int(rng.choice([2, 4]))
        y = rng.standard_normal(6 * nf).astype(np.float32)
        spec = np.asarray(O.stft(y, n_fft=nf, hop_length=hp)).astype(np.complex64)       # both sides invert the same spectrogram
        norm = bool(rng.integers(0, 2))
        ib = O.istft(spec.T, hop_length=hp, win_length=nf, normalized=norm)
        worst["istft"] = max(worst["istft"], tape.err(lambda: dsp.istft(numpy_mlx_shim.array(spec.T), hop_length=hp, win_length=nf, normalized=norm), ib))
        sr = int(rng.choice([16000, 22050, 24000, 44100]))
        mk = dict(sample_rate=sr, n_fft=int(rng.choice([256, 400, 1024])), n_mels=int(rng.choice([20, 40, 80, 128])), f_min=float(rng.choice([0.0, 50.0])),
                  f_max=float(rng.choice([sr / 2, sr / 2 - 1000.0])), norm=[None, "slaney"][int(rng.integers(0, 2))], mel_scale=str(rng.choice(["htk", "slaney"])))
        worst["mel"] = max(worst["mel"], tape.err(lambda: dsp.mel_filters(**mk), O.mel_filters(**mk)))
        print("dsp", kw, "| istft", nf, hp, norm, "| mel", mk["sample_rate"], mk["n_mels"], mk["norm"], mk["mel_scale"])
    # interpolate (tts/models/interpolate.py): nearest / linear, align_corners on / off / None, up- and down-scaling incl. the 300x of Kokoro's source
    sys.path.insert(0, HERE)
    import numpy_mlx_nn as nn_shim
    core64, _ = nn_shim.install(precise=True)
    if tape.reference:
        interp = load(os.path.join(REF, "tts", "models", "interpolate.py"), "ref_interpolate_live")
    worst["interp"] = 0.0
    for seed in range(6 * n):
        rng = np.random.default_rng(6000 + seed)
        x = rng.standard_normal((int(rng.integers(1, 3)), int(rng.integers(1, 4)), int(rng.integers(2, 700))))
        mode = str(rng.choice(["nearest", "linear"]))
        ac = [None, False, True][int(rng.integers(0, 3))] if mode == "linear" else None
        if rng.random() < 0.5:
            kw = dict(scale_factor=float(rng.choice([2.0, 0.5, 1 / 3, 3.0, 300.0, 1 / 300, 1.7])))
        else:
            kw = dict(size=int(rng.integers(1, 900)))
        if x.shape[-1] * kw.get("scale_factor", 1.0) > 40000:
            x = x[..., :100]
        b = O.interpolate(x, mode=mode, align_corners=ac, **kw)
        worst["interp"] = max(worst["interp"], tape.err(lambda: interp.interpolate(core64.array(x), mode=mode, align_corners=ac, **kw), b))
    tape.close()
    print(worst)
    assert worst["interp"] < 1e-12, worst
    assert worst["stft"] < 2e-4 and worst["istft"] < 5e-5 and worst["mel"] < 5e-6 and worst["window"] < 1e-6, worst
    print("LIVE OK", worst)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--live":
        live(int(sys.argv[2]))
    else:
        main()
