"""The committed fixtures under tests/golden/ are outputs of the reference's own source.  Where that source is present (REF in the
generators), every generator is re-run into a scratch directory and its output compared with the committed file -- so a fixture can
never drift from the code that is supposed to have produced it; without it those tests skip.  The random-configuration comparisons
of the oracle with the reference run everywhere, against the reference results recorded in tests/golden/*_live_golden.npz."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROOT = os.path.dirname(os.path.dirname(HERE))
GENERATORS = {"make_cache_golden.py": "cache_golden.npz", "make_codec_golden.py": "codec_golden.npz", "make_config_golden.py": "config_golden.json",
              "make_dsp_golden.py": "dsp_golden.npz", "make_kokoro_golden.py": "kokoro_golden.npz", "make_qwen3_golden.py": "qwen3_golden.npz",
              "make_resample_golden.py": "resample_golden.npz", "make_sanitize_golden.py": "sanitize_golden.json",
              "make_whisper_golden.py": "whisper_golden.npz"}


def _json_close(a, b):
    if isinstance(a, float) or isinstance(b, float):
        return isinstance(a, (int, float)) and isinstance(b, (int, float)) and (a == b or (a != a and b != b) or abs(a - b) <= 1e-9 * max(1.0, abs(b)))
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(_json_close(a[k], b[k]) for k in a)
    if isinstance(a, list):
        return isinstance(b, list) and len(a) == len(b) and all(_json_close(x, y) for x, y in zip(a, b))
    return a == b


@pytest.mark.skipif(not os.path.isdir("/root/reference/mlx_audio"), reason="the reference source is only present in the build container")
@pytest.mark.parametrize("generator", sorted(GENERATORS))
def test_fixture_is_what_the_reference_code_produces(generator, tmp_path):
    env = dict(os.environ, GOLDEN_OUT=str(tmp_path), OMP_NUM_THREADS="4")
    r = subprocess.run([sys.executable, os.path.join(HERE, generator)], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    name = GENERATORS[generator]
    if name.endswith(".json"):
        assert json.load(open(tmp_path / name)) == json.load(open(os.path.join(HERE, name)))
        return
    new, old = np.load(tmp_path / name), np.load(os.path.join(HERE, name))
    assert sorted(new.files) == sorted(old.files)
    for k in old.files:
        a, b = new[k], old[k]
        if a.dtype.kind == "U" and b.dtype.kind == "U":       # JSON text (the Whisper generate() results): floats to 1e-9, everything else exactly
            assert _json_close(json.loads(str(a)), json.loads(str(b))), k
            continue
        assert a.dtype == b.dtype and a.shape == b.shape, k
        if a.dtype.kind in "fc":
            fin = np.isfinite(b)
            assert np.array_equal(np.isfinite(a), fin) and np.array_equal(a[~fin], b[~fin], equal_nan=True), k
            scale = max(1.0, float(np.abs(b[fin]).max())) if fin.any() else 1.0
            assert np.abs(a[fin] - b[fin]).max(initial=0.0) <= 1e-12 * scale, k
        else:
            assert np.array_equal(a, b), k


@pytest.mark.parametrize("generator,n", [("make_dsp_golden.py", 12), ("make_whisper_golden.py", 4), ("make_qwen3_golden.py", 4), ("make_codec_golden.py", 5), ("make_kokoro_golden.py", 2)])
def test_oracle_agrees_with_the_reference_code_on_random_configurations(generator, n):
    """Beyond the committed fixtures: ``--live N`` draws N random configurations (head counts, GQA ratios, MRoPE sections, code-book counts,
    stride lists, depthwise / noise switches, attention contexts, kernel sizes; for Kokoro random utterances, styles, speeds and weight
    seeds), runs the reference's classes through the NumPy stand-in and the oracle side by side, and requires 1e-9 (identical integer
    results).  This is what guards the oracle's generality between the small fixture configurations and the full-size ones the CUDA path is
    tested against; it found two hard-coded assumptions (decoder layer indices for four upsampling stages, SNAC's depthwise stem).
    ``--replay`` draws the same configurations and runs the oracle against the reference's results as ``--live N --record`` stored them
    (tests/golden/live_tape.py), so it needs no reference source."""
    r = subprocess.run([sys.executable, os.path.join(HERE, generator), "--live", str(n), "--replay"], cwd=ROOT, env=dict(os.environ, OMP_NUM_THREADS="4"),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "LIVE OK" in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])
