"""What the original chunkflow computed on the inputs the pinning tests build, so that those tests compare against it
without the original project at hand.  `tests/golden/make_golden_reference.py` runs the original project and records;
the tests check.  The same calls do both:

    pins.exact(key, array)    bit-exact: shape, dtype and the sha256 of the bytes (C order) are stored
    pins.close(key, array)    with a tolerance: the values are stored (a fixed, seeded sample of large arrays)
    pins.value(key, obj)      anything JSON can hold (offsets, attribute values, option tables, signatures)
"""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
JSON_PATH = os.path.join(GOLDEN, "reference_pins.json")
NPZ_PATH = os.path.join(GOLDEN, "reference_pins.npz")
CLOSE_SAMPLE = 1 << 13     # values kept of an array compared with a tolerance, when it has more
REQUIRED = "<required>"    # the default of a parameter without one, in recorded signatures


def plain(obj):
    """JSON round trip: tuples become lists, numpy scalars and arrays become numbers and lists."""
    def default(o):
        if isinstance(o, (np.integer, np.floating, np.bool_)):
            return o.item()
        if isinstance(o, np.ndarray):
            return o.tolist()
        raise TypeError(type(o))
    return json.loads(json.dumps(obj, default=default))


def _sample_index(size):
    return np.sort(np.random.default_rng(20261017).choice(size, CLOSE_SAMPLE, replace=False)) if size > CLOSE_SAMPLE else None


class Pins:
    def __init__(self, record=False):
        self.record = record
        if record:
            self.meta, self.arrays = {}, {}
        else:
            with open(JSON_PATH) as f:
                self.meta = json.load(f)
            with np.load(NPZ_PATH) as z:
                self.arrays = {k: z[k] for k in z.files}

    def _stored(self, key):
        assert key in self.meta, f"no reference output recorded for {key!r}: rerun tests/golden/make_golden_reference.py"
        return self.meta[key]

    def exact(self, key, a):
        a = np.ascontiguousarray(a)
        got = {"shape": list(a.shape), "dtype": a.dtype.str, "sha256": hashlib.sha256(a.tobytes()).hexdigest()}
        if self.record:
            self.meta[key] = got
        else:
            want = self._stored(key)
            assert got["shape"] == want["shape"] and got["dtype"] == want["dtype"], (key, got, want)
            assert got["sha256"] == want["sha256"], f"{key}: differs from the reference's output"

    def close(self, key, a, atol=0.0):
        a = np.asarray(a)
        idx = _sample_index(a.size)
        values = a.reshape(-1) if idx is None else a.reshape(-1)[idx]
        if self.record:
            self.meta[key] = {"shape": list(a.shape), "dtype": a.dtype.str, "sampled": idx is not None}
            self.arrays[key] = values
        else:
            want = self._stored(key)
            assert list(a.shape) == want["shape"] and a.dtype.str == want["dtype"], (key, a.shape, a.dtype, want)
            np.testing.assert_allclose(values, self.arrays[key], rtol=0, atol=atol, err_msg=key)

    def value(self, key, obj):
        obj = plain(obj)
        if self.record:
            self.meta[key] = obj
        else:
            assert obj == self._stored(key), (key, obj, self.meta[key])
        return obj

    def get(self, key):
        """A recorded value, for tests that compare against it with more than equality."""
        return self._stored(key)

    def save(self, **info):
        self.meta.update({f"_{k}": v for k, v in info.items()})
        with open(JSON_PATH, "w") as f:     # one entry per line
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(self.meta.items())) + "\n}\n")
        np.savez_compressed(NPZ_PATH, **self.arrays)
