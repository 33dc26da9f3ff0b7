"""What the original chunkflow's ``Segmentation.evaluate`` computed on the cases of tests/test_evaluate_segmentation.py, kept
apart from the other pins in tests/golden/evaluate_pins.{json,npz} (recorded by tests/golden/make_golden_evaluate.py).
Same calls and file format as :class:`reference_pins.Pins`, other files."""
import json
import os

import numpy as np

from reference_pins import GOLDEN, Pins

JSON_PATH = os.path.join(GOLDEN, "evaluate_pins.json")
NPZ_PATH = os.path.join(GOLDEN, "evaluate_pins.npz")


class EvaluatePins(Pins):
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
        assert key in self.meta, f"no reference output recorded for {key!r}: rerun tests/golden/make_golden_evaluate.py"
        return self.meta[key]

    def save(self, **info):
        self.meta.update({f"_{k}": v for k, v in info.items()})
        with open(JSON_PATH, "w") as f:     # one entry per line
            f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(self.meta.items())) + "\n}\n")
        np.savez_compressed(NPZ_PATH, **self.arrays)
