"""Results of the unmodified reference library on the problems of the comparison tests, stored under tests/golden so
that every comparison runs wherever the repository is checked out, with or without the reference's sources.

A test asks for a result by a key that names the run, together with the function that computes it from a library:

    b = reference("rosenbrock/24", lambda lib: run(lib, ...))

The stored result is returned and the function is not called.  A result is a dict or a tuple of ints, floats, strings
and float arrays.  reference_runs.json holds every result, floats exactly (float.hex), arrays as a slice of the one
float64 array in reference_runs.npz.  To regenerate the files, build the reference into oracle/_ref
(oracle/Makefile: `make -C oracle ref REF=<the reference's source tree>`) and run

    NLOPT_B200_RECORD_REFERENCE=1 python -m pytest tests

which runs only the tests that use the `reference` fixture, calls each function on oracle/_ref/libnlopt_ref.so
(comparing against it live), and writes every result it produced into the files.  On a machine without a GPU the
GPU-marked comparisons record their reference side and then skip."""
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RUNS = os.path.join(GOLDEN, "reference_runs.json")
ARRAYS = os.path.join(GOLDEN, "reference_runs.npz")
RECORDING = os.environ.get("NLOPT_B200_RECORD_REFERENCE") == "1"


def _encode(v, arrays):
    if isinstance(v, (bool, np.bool_, int, np.integer)):
        return int(v)
    if isinstance(v, (float, np.floating)):
        return {"float": float(v).hex()}
    if isinstance(v, str):
        return v
    a = np.asarray(v, dtype=np.float64).ravel()
    arrays.append(a)
    return {"array": [sum(x.size for x in arrays[:-1]), a.size]}


def _decode(v, values):
    if isinstance(v, dict):
        if "float" in v:
            return float.fromhex(v["float"])
        off, size = v["array"]
        return values[off:off + size].copy()
    return v


class Store:
    """The stored results (replay), or the live reference library and the results recorded from it."""

    def __init__(self, lib=None):
        self.lib = lib
        self.recorded = {}
        self.stored, self.values = {}, np.empty(0)
        if os.path.exists(RUNS):
            with open(RUNS) as f:
                self.stored = json.load(f)
            with np.load(ARRAYS) as z:
                self.values = z["values"]

    def get(self, key, compute):
        if self.lib is not None:
            result = compute(self.lib)
            self.recorded[key] = result
            return result
        if key not in self.stored:
            raise KeyError(f"no stored reference result {key!r} in {RUNS}; regenerate it (see tests/reference_runs.py)")
        r = self.stored[key]
        if isinstance(r, list):
            return tuple(_decode(v, self.values) for v in r)
        return {k: _decode(v, self.values) for k, v in r.items()}

    def save(self):
        if not self.recorded:
            return
        runs = {k: (tuple(_decode(v, self.values) for v in r) if isinstance(r, list) else
                    {f: _decode(v, self.values) for f, v in r.items()}) for k, r in self.stored.items()}
        runs.update(self.recorded)
        arrays, out = [], {}
        for key in sorted(runs):
            r = runs[key]
            out[key] = ([_encode(v, arrays) for v in r] if isinstance(r, tuple) else
                        {f: _encode(v, arrays) for f, v in r.items()})
        with open(RUNS, "w") as f:
            json.dump(out, f, indent=0, sort_keys=True)
            f.write("\n")
        np.savez_compressed(ARRAYS, values=np.concatenate(arrays) if arrays else np.empty(0))
