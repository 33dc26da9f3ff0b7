"""Record what the REAL reference's ``Segmentation.evaluate`` computes on the cases of tests/test_evaluate_segmentation.py
(its scores, its printout and its contingency table) and the option tables of its `load-npy` and `evaluate-segmentation`
commands into tests/golden/evaluate_pins.{json,npz}.  Needs the reference tree (oracle/reference_harness.py says where it is
looked for; oracle/evaluation_harness.py which missing packages are stubbed):

    python tests/golden/make_golden_evaluate.py
"""
import ast
import io
import os
import re
import sys
import warnings
from contextlib import redirect_stdout

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from oracle import evaluation_harness as E, reference_harness as H  # noqa: E402
from evaluate_pins import EvaluatePins  # noqa: E402
import test_evaluate_segmentation as T  # noqa: E402


def cli_table(src, command):
    """[flags, literal default or None, required] per option of the LAST definition of `command` in flow/flow.py (the one
    click keeps when a name is registered twice)."""
    seg = src[src.rindex(f"@main.command('{command}')"):]
    seg = seg[:seg.index("\ndef ")]
    opts = []
    for m in re.finditer(r"@click\.option\((.*?)\)\s*(?=@click\.option|@operator|@generator|@main|$)", seg, re.S):
        body = m.group(1)
        flags = re.findall(r"""['"](-{1,2}[A-Za-z][\w/-]*)['"]""", body.split("help=")[0])
        default = re.search(r"default=(\([^)]*\)|[^,\s)]+)", body)
        try:
            value = ast.literal_eval(default.group(1)) if default else None
        except (ValueError, SyntaxError):
            value = None     # a name such as DEFAULT_CHUNK_NAME
        opts.append([flags, value, "required=True" in body])
    return opts


def main():
    warnings.simplefilter("ignore")
    Segmentation, evaluate = E.import_reference_evaluation()
    pins = EvaluatePins(record=True)
    for i, (seg, gt, thr) in enumerate(T.evaluate_cases()):
        out = io.StringIO()
        with redirect_stdout(out):
            r = Segmentation(seg.copy()).evaluate(gt.copy(), size_threshold=thr)
        assert list(r) == list(T.O.SCORE_KEYS)
        pins.value(f"evaluate/{i}/scores", {k: (list(v) if k == "edit_distance" else v) for k, v in r.items()})
        pins.value(f"evaluate/{i}/printed", out.getvalue())
        t = evaluate.contingency_table(seg.astype(np.uint64), gt.astype(np.uint64), norm=False).tocoo()
        t.sum_duplicates()
        keep = t.data != 0
        order = np.lexsort((t.col[keep], t.row[keep]))
        for name, a in (("seg", t.row[keep]), ("gt", t.col[keep]), ("count", t.data[keep])):
            pins.close(f"evaluate/{i}/table_{name}", np.asarray(a, np.float64)[order])
    with open(os.path.join(H.REFERENCE_ROOT, "chunkflow", "flow", "flow.py")) as f:
        src = f.read()
    for command in ("load-npy", "evaluate-segmentation"):
        pins.value(f"cli/{command}", cli_table(src, command))
    pins.save(numpy=np.__version__)
    print("reference outputs recorded:", len(pins.meta), "entries")


if __name__ == "__main__":
    main()
