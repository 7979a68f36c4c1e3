"""Record / replay of the reference side of the generators' ``--live N`` comparisons.

``--live N`` runs the reference's classes and the oracle side by side.  ``--live N --record`` does the same and stores, in call order,
everything the comparison takes from the reference: small values whole (parameter manifests, integer results, shapes), and for
every float result its shape, its non-finite pattern, its sum and a seeded sample of its values.  ``--live N --replay`` draws the
same random configurations and runs the oracle side against that record, so the comparison runs without the reference source.

On replay a float comparison is the larger of the sampled element-wise error and the error of the mean over the finite elements
(the mean of the differences is bounded by their maximum, so one tolerance covers both)."""
import json
import os

import numpy as np

SAMPLE = 12          # sampled elements per float result


def _path(name):
    return os.path.join(os.environ.get("GOLDEN_OUT", os.path.dirname(os.path.abspath(__file__))), f"{name}_live_golden.npz")


def _runs(mask):
    """[[start, stop], ...] of the True runs of a flat bool array (suppressed logits come in blocks)."""
    d = np.diff(np.concatenate([[0], mask.astype(np.int8), [0]]))
    return np.stack([np.flatnonzero(d == 1), np.flatnonzero(d == -1)], axis=1).tolist()


def _jsonable(v):
    if isinstance(v, np.ndarray):
        return v.tolist()
    if isinstance(v, (np.integer, np.bool_)):
        return v.item()
    if isinstance(v, (list, tuple)):
        return [_jsonable(x) for x in v]
    return v


class Tape:
    def __init__(self, name, n, argv):
        self.name, self.n, self.items, self.pos = name, n, [], 0
        self.mode = "replay" if "--replay" in argv else "record" if "--record" in argv else "live"
        if self.mode == "replay":
            g = np.load(_path(name))
            assert int(g["n"]) == n, f"{_path(name)} holds {int(g['n'])} configurations, not {n}"
            self.items = json.loads(str(g["tape"]))

    @property
    def reference(self):
        """True when the reference runs (live or record)."""
        return self.mode != "replay"

    def _next(self, kind):
        assert self.pos < len(self.items), "the record ends early: it was made by another version of this generator"
        item = self.items[self.pos]
        self.pos += 1
        assert item[0] == kind, (self.pos, kind, item[0])
        return item[1]

    def value(self, fn):
        """A reference-side value stored whole (JSON: lists, ints, strings); ``fn`` only runs when the reference does."""
        if self.mode == "replay":
            return self._next("v")
        v = _jsonable(fn())
        if self.mode == "record":
            self.items.append(["v", v])
        return v

    def err(self, fn, got, same_nonfinite=False, sample=SAMPLE):
        """Max |reference - got| over the positions where the reference is finite; ``same_nonfinite`` also requires both to be
        non-finite at the same positions.  ``fn`` returns the reference array and only runs when the reference does; ``sample``
        elements of it are recorded.  A NaN difference is reported as inf."""
        got = np.asarray(got)
        if self.mode == "replay":
            r = self._next("a")
            assert list(got.shape) == r["shape"], (got.shape, r["shape"])
            flat = got.reshape(-1)
            fin = np.ones(flat.size, bool)
            for a, b in r["nonfinite"]:
                fin[a:b] = False
            if same_nonfinite:
                assert np.array_equal(np.isfinite(flat), fin), "non-finite pattern differs"
            idx = np.asarray(r["idx"], dtype=np.int64)
            want = np.asarray(r["re"]) + (1j * np.asarray(r["im"]) if "im" in r else 0)
            e = float(np.abs(flat[idx] - want).max(initial=0.0))
            n_fin = int(fin.sum())
            if n_fin:
                s = r["sum_re"] + (1j * r["sum_im"] if "im" in r else 0)
                e = max(e, float(abs(flat[fin].sum() - s)) / n_fin)
            return e if e == e else float("inf")
        ref = np.asarray(fn())
        assert ref.shape == got.shape, (ref.shape, got.shape)
        fin = np.isfinite(ref)
        if same_nonfinite:
            assert np.array_equal(np.isfinite(got), fin), "non-finite pattern differs"
        if self.mode == "record":
            flat, ffin = ref.reshape(-1), fin.reshape(-1)
            pos = np.flatnonzero(ffin)
            idx = np.sort(np.random.default_rng(len(self.items)).choice(pos, min(sample, pos.size), replace=False))
            r = {"shape": list(ref.shape), "nonfinite": _runs(~ffin), "idx": idx.tolist(),
                 "re": flat[idx].real.tolist(), "sum_re": float(flat[ffin].sum().real)}
            if np.iscomplexobj(ref):
                r["im"], r["sum_im"] = flat[idx].imag.tolist(), float(flat[ffin].sum().imag)
            self.items.append(["a", r])
        e = float(np.abs(ref[fin] - got[fin]).max(initial=0.0))
        return e if e == e else float("inf")          # a NaN would pass every max() and < tolerance unnoticed

    def close(self):
        if self.mode == "record":
            np.savez_compressed(_path(self.name), n=self.n, tape=json.dumps(self.items))
        if self.mode == "replay":
            assert self.pos == len(self.items), "the record holds more comparisons than were replayed"
