"""Import the REAL reference's ``Segmentation`` and gala ``evaluate`` module (TEST INFRASTRUCTURE, used by
tests/golden/make_golden_evaluate.py only).

``chunk/segmentation.py`` and ``lib/gala/evaluate.py`` import h5py, skimage, sklearn, fastremap and cloudfiles, which are not
installed offline; on top of the stubs of ``reference_harness.import_reference`` this registers empty stand-ins for them.
Only works where the reference tree exists (``reference_harness.REFERENCE_ROOT``).
"""
import sys
import types

import numpy as np

from oracle import reference_harness


def _stub(name, **attrs):
    m = sys.modules.get(name) or types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def relabel_sequential(label_field):
    """Stand-in for ``skimage.segmentation.relabel_sequential`` with its default offset of 1: sorted non-zero ids -> 1..K,
    0 kept.  ``Segmentation.evaluate`` uses it only in the edit distance (evaluate.py:194-209), to renumber both volumes
    before their contingency table is built; that table is then the same up to a renaming of rows and columns, and so is
    the edit distance."""
    ids = np.unique(label_field)
    ids = ids[ids != 0]
    out = np.zeros(label_field.shape, np.int64)
    nz = label_field != 0
    out[nz] = np.searchsorted(ids, label_field[nz]) + 1
    return out, None, None


def import_reference_evaluation():
    """Returns (Segmentation, gala evaluate module) of the real reference."""
    reference_harness.import_reference()
    sk = _stub("skimage")
    sk.segmentation = _stub("skimage.segmentation", relabel_sequential=relabel_sequential)
    _stub("sklearn")
    _stub("sklearn.metrics", precision_recall_curve=lambda *a, **k: None)
    _stub("fastremap")
    _stub("cloudfiles", CloudFiles=type("CloudFiles", (), {}))
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        from chunkflow.chunk.segmentation import Segmentation
        from chunkflow.lib.gala import evaluate
    return Segmentation, evaluate
