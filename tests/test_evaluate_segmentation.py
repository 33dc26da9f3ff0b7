"""`evaluate-segmentation`: the oracle (oracle/evaluation_oracle.py) against what the real reference's
``Segmentation.evaluate`` computed on seeded cases (tests/golden/evaluate_pins.json, recorded by
tests/golden/make_golden_evaluate.py), the device code on the host through a one-thread shim
(tests/host_emulation/evaluate_emulation.cpp) against the oracle, and on the GPU the device scores and pair table against
the oracle.  RI, ARI, FM and the edit distance must be equal (NaN included), VI within 1e-12.
"""
import ctypes as C
import io
import math
import os
import shutil
import subprocess
from contextlib import redirect_stdout

import numpy as np
import pytest

from conftest import ROOT, has_gpu
from oracle import evaluation_oracle as O

gpu = pytest.mark.gpu
VI_ATOL = 1e-12


def evaluate_cases():
    """-> list of (seg, gt, size_threshold), both uint32 (z, y, x)."""
    rng = np.random.default_rng(20261017)
    cases = []

    def add(seg, gt, thr):
        cases.append((np.ascontiguousarray(seg, np.uint32), np.ascontiguousarray(gt, np.uint32), thr))

    thresholds = (0, 10, 1000, 12.5)
    for i in range(16):   # random labels: 1 .. thousands of ids, with and without background
        shape = tuple(int(v) for v in rng.integers(1, 24, 3))
        ks, kg = (int(v) for v in rng.choice([1, 2, 3, 7, 40, 300, 3000], 2))
        seg = rng.integers(0, ks, shape)
        gt = rng.integers(0, kg, shape)
        if i % 4 == 1:
            seg[rng.random(shape) < 0.8] = 0   # heavy background
        if i % 4 == 2:
            seg, gt = seg + 1, gt + 1          # no background
        add(seg, gt, thresholds[i % 4])
    for i in range(6):    # blocky segmentations: large overlaps, so that the edit distance's threshold matters
        shape = (8, 24, 24)
        z, y, x = np.indices(shape)
        seg = (z // 4) * 9 + (y // 8) * 3 + x // 8 + 1
        gt = ((z + i) // 4) * 16 + ((y + 2 * i) // 6) * 4 + (x + i) // 6
        if i % 2:
            gt[rng.random(shape) < 0.1] = 0
        add(seg, gt, thresholds[i % 4])
    one = np.ones((1, 1, 1))
    add(one, one, 1000)                                    # a single voxel: RI = ARI = FM = NaN, VI = 0
    add(0 * one, one, 0)
    add(np.zeros((4, 5, 6)), rng.integers(0, 4, (4, 5, 6)), 1000)   # all-zero segmentation: VI = NaN
    add(rng.integers(0, 4, (4, 5, 6)), np.zeros((4, 5, 6)), 0)
    add(np.zeros((3, 3, 3)), np.zeros((3, 3, 3)), 1000)
    s = rng.integers(1, 5, (3, 5, 8))
    add(s, s, 0)                                           # against itself: 120 voxels, edit distance -K
    add(np.full((2, 9, 7), 5), rng.integers(0, 6, (2, 9, 7)), 10)
    add(rng.integers(0, 2 ** 20, (6, 7, 8)), rng.integers(0, 2 ** 20, (6, 7, 8)), 0)   # every pair distinct
    return cases


def _same(got, want):
    return (isinstance(got, float) and isinstance(want, float) and math.isnan(got) and math.isnan(want)) or got == want


def assert_scores(got, want, vi_atol=VI_ATOL, rtol=0.0):
    assert list(got) == list(O.SCORE_KEYS)
    for k in O.SCORE_KEYS:
        g, w = got[k], want[k]
        if k == "edit_distance":
            assert tuple(float(v) for v in g) == tuple(float(v) for v in w), (k, g, w)
        elif k == "variation_of_information":
            assert (math.isnan(g) and math.isnan(w)) or abs(float(g) - float(w)) <= vi_atol + rtol * abs(float(w)), (k, g, w)
        elif rtol:
            assert (math.isnan(g) and math.isnan(w)) or abs(float(g) - float(w)) <= rtol * abs(float(w)), (k, g, w)
        else:
            assert _same(float(g), float(w)), (k, g, w)


@pytest.fixture(scope="module")
def evaluate_pins():
    from evaluate_pins import EvaluatePins
    return EvaluatePins()


def recorded(pins, i):
    r = pins.get(f"evaluate/{i}/scores")
    r = {k: (tuple(v) if k == "edit_distance" else float(v)) for k, v in r.items()}
    return r


# ------------------------------------------------------------------------------------------------------------
# CPU: the oracle against the recorded reference
# ------------------------------------------------------------------------------------------------------------
def test_oracle_matches_the_reference(evaluate_pins):
    cases = evaluate_cases()
    assert len(cases) >= 30
    for i, (seg, gt, thr) in enumerate(cases):
        want = recorded(evaluate_pins, i)
        got = O.evaluate(seg, gt, thr)
        assert_scores(got, want)
        assert O.format_scores(got) == evaluate_pins.get(f"evaluate/{i}/printed"), i


def test_oracle_pair_table_matches_the_reference_table(evaluate_pins):
    for i, (seg, gt, _) in enumerate(evaluate_cases()):
        s, g, c = O.contingency_pairs(seg, gt)
        for name, a in (("seg", s), ("gt", g), ("count", c)):
            evaluate_pins.close(f"evaluate/{i}/table_{name}", a.astype(np.float64))


def test_product_scores_and_printout_equal_the_oracle():
    """The host half of the product (scores from the sums, the printout) on the oracle's sums, as exact fixed point."""
    from fractions import Fraction
    from chunkflow_b200 import _native
    from chunkflow_b200.chunk.segmentation import format_scores, scores_from_sums
    for seg, gt, thr in evaluate_cases():
        s = O.sums(seg, gt, thr)
        native = _native.ContingencySums()
        for k in ("voxels", "entries", "sum_sq_pairs", "sum_sq_seg", "sum_sq_gt", "nonzero_voxels", "seg_labels", "pairs_over_threshold"):
            setattr(native, k, s[k])
        for k in ("xlogx_pairs", "xlogx_seg", "xlogx_gt"):
            f = int(Fraction(s[k]) * 2 ** 62)
            getattr(native, k)[:] = [f & (2 ** 64 - 1), f >> 64]
        got = scores_from_sums(native)
        assert_scores(got, O.evaluate(seg, gt, thr))
        assert format_scores(got) == O.format_scores(got)


def test_cli_options_match_the_reference_source(evaluate_pins):
    """The two new commands keep the reference's flags, defaults and required-ness (flow/flow.py:1321-1341, 1519-1542)."""
    from chunkflow_b200.flow import cli
    for command, obj in (("load-npy", cli.load_npy), ("evaluate-segmentation", cli.evaluate_segmentation)):
        mine = {}
        for p in obj.params:
            for o in p.opts:
                mine[o] = p
        ref = evaluate_pins.get(f"cli/{command}")
        assert len(ref) == len(obj.params), command
        for flags, default, required in ref:
            for f in flags:
                assert f in mine, (command, f)
            p = mine[flags[0]]
            got = p.default
            if isinstance(default, list):
                default, got = tuple(default), tuple(got)
            assert got == default or (default is None and command == "load-npy" and flags[0] == "--output-name"), (command, flags)
            assert bool(p.required) == required, (command, flags)
        if command == "load-npy":
            assert mine["--output-name"].default == "chunk"   # the reference's DEFAULT_CHUNK_NAME (lib/flow.py:21)


def test_load_npy_command(tmp_path):
    from chunkflow_b200.flow import cli
    a = np.arange(60, dtype=np.uint16).reshape(3, 4, 5)
    path = tmp_path / "gt.npy"
    np.save(path, a)
    tasks = cli.main.main(["create-chunk", "--size", "3", "4", "5", "load-npy", "-f", str(path), "-t", "1", "2", "3", "-s", "4", "4", "40",
                           "-o", "groundtruth"], standalone_mode=False)
    gt = tasks[0]["groundtruth"]
    assert np.array_equal(gt.array, a) and tuple(gt.voxel_offset) == (1, 2, 3) and tuple(gt.voxel_size) == (4, 4, 40)


def test_segmentation_checks_its_input():
    from chunkflow_b200.chunk.segmentation import Segmentation
    from chunkflow_b200 import Chunk
    with pytest.raises(ValueError):
        Segmentation(np.zeros((1, 2, 3, 4), np.uint32))
    with pytest.raises(TypeError):
        Segmentation(np.zeros((2, 3, 4), np.float32))
    s = Segmentation.from_chunk(Chunk(np.zeros((2, 3, 4), np.int64), voxel_offset=(1, 2, 3)))
    assert tuple(s.voxel_offset) == (1, 2, 3)
    with pytest.raises(ValueError):
        s.evaluate(np.zeros((2, 3, 5), np.uint32))
    with pytest.raises(TypeError):
        s.evaluate(np.zeros((2, 3, 4), np.float64))


def test_segmentation_evaluate_needs_a_gpu(monkeypatch):
    import torch
    from chunkflow_b200.chunk.segmentation import Segmentation
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    with pytest.raises(RuntimeError, match="CUDA"):
        Segmentation(np.ones((2, 3, 4), np.uint32)).evaluate(np.ones((2, 3, 4), np.uint32))


# ------------------------------------------------------------------------------------------------------------
# the device code on the host (one-thread CUDA shim)
# ------------------------------------------------------------------------------------------------------------
class _Sums(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("voxels", "entries", "sum_sq_pairs", "sum_sq_seg", "sum_sq_gt", "nonzero_voxels",
                                          "seg_labels", "pairs_over_threshold")] + \
               [(n, C.c_uint64 * 2) for n in ("xlogx_pairs", "xlogx_seg", "xlogx_gt")]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("ev_emu") / "libev_emu.so"
    src = os.path.join(ROOT, "tests", "host_emulation", "evaluate_emulation.cpp")
    subprocess.run([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", src, "-o", str(out)], check=True)
    lib = C.CDLL(str(out))
    lib.emu_contingency.restype = C.c_int64
    lib.emu_contingency.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int64, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.POINTER(_Sums)]
    return lib


def _emu_run(lib, seg, gt, thr, slots=1 << 12):
    seg, gt = np.ascontiguousarray(seg), np.ascontiguousarray(gt)
    os_, og, oc = (np.empty(slots, np.uint64) for _ in range(3))
    sums = _Sums()
    e = lib.emu_contingency(seg.ctypes.data, int(seg.dtype.itemsize == 8), gt.ctypes.data, int(gt.dtype.itemsize == 8), seg.size, slots,
                            float(thr), os_.ctypes.data, og.ctypes.data, oc.ctypes.data, C.byref(sums))
    return e, (os_[:max(e, 0)], og[:max(e, 0)], oc[:max(e, 0)]), sums


def _fixed(v):
    return (int(v[0]) | (int(v[1]) << 64)) / 2 ** 62


def test_device_code_on_the_host_equals_the_oracle(emu):
    for i, (seg, gt, thr) in enumerate(evaluate_cases()):
        if i % 2:   # the 64-bit loads on half the cases
            seg = seg.astype(np.uint64) * np.uint64(2 ** 32 + 1)
        e, table, sums = _emu_run(emu, seg, gt, thr, slots=1 << 17)
        want = O.contingency_pairs(seg, gt)
        assert e == want[0].size, i
        for a, b in zip(table, want):
            assert np.array_equal(a, b), i
        s = O.sums(seg, gt, thr)
        for k in ("voxels", "entries", "sum_sq_pairs", "sum_sq_seg", "sum_sq_gt", "nonzero_voxels", "seg_labels", "pairs_over_threshold"):
            assert getattr(sums, k) == s[k], (i, k)
        for k in ("xlogx_pairs", "xlogx_seg", "xlogx_gt"):
            assert abs(_fixed(getattr(sums, k)) - s[k]) <= 1e-9 * max(1.0, s[k]), (i, k)


def test_device_code_on_the_host_reports_a_full_table(emu):
    rng = np.random.default_rng(3)
    seg = rng.integers(0, 1000, (4, 8, 8)).astype(np.uint32)
    e, _, _ = _emu_run(emu, seg, seg, 0, slots=64)
    assert e == -1
    e, _, _ = _emu_run(emu, seg, seg, 0, slots=2048)
    assert e == np.unique(seg).size


# ------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------
def _device(a):
    from chunkflow_b200.chunk.device import DeviceChunk
    from chunkflow_b200.chunk.segmentation import label_array
    return DeviceChunk.from_labels(label_array(a, "labels"))


DTYPES = [(np.uint32, np.uint32), (np.uint32, np.uint64), (np.uint64, np.uint32), (np.uint64, np.uint64)]


@gpu
@pytest.mark.parametrize("sdt,gdt", DTYPES, ids=lambda d: np.dtype(d).name)
def test_device_scores_equal_the_reference(evaluate_pins, sdt, gdt):
    assert has_gpu()
    for i, (seg, gt, thr) in enumerate(evaluate_cases()):
        got = _device(seg.astype(sdt)).evaluate(_device(gt.astype(gdt)), size_threshold=thr)
        assert_scores(got, recorded(evaluate_pins, i))


@gpu
def test_segmentation_evaluate_prints_and_returns_the_reference_dict(evaluate_pins):
    from chunkflow_b200.chunk.segmentation import Segmentation
    for i, (seg, gt, thr) in enumerate(evaluate_cases()):
        for s, g in ((seg.astype(np.uint16) if seg.max() < 2 ** 16 else seg, gt.astype(np.int64)),):
            f = io.StringIO()
            with redirect_stdout(f):
                got = Segmentation(s).evaluate(g, size_threshold=thr)
            assert_scores(got, recorded(evaluate_pins, i))
            assert f.getvalue() == evaluate_pins.get(f"evaluate/{i}/printed"), i


@gpu
def test_device_pair_table_equals_numpy_unique():
    rng = np.random.default_rng(5)
    for seg, gt, _ in evaluate_cases()[::3] + [(rng.integers(0, 50, (33, 65, 67)), rng.integers(0, 9, (33, 65, 67)), 0)]:
        got = _device(seg.astype(np.uint32)).contingency_table(_device(gt.astype(np.uint64)))
        for a, b in zip(got, O.contingency_pairs(seg, gt)):
            assert a.dtype == np.uint64 and np.array_equal(a, b)


@gpu
def test_large_ids_score_like_their_dense_relabelling():
    ids = np.array([0, 2 ** 32 - 1, 2 ** 63, 2 ** 64 - 1, 10 ** 12], np.uint64)
    rng = np.random.default_rng(7)
    for shape in ((5, 6, 7), (16, 33, 31)):
        a, b = rng.integers(0, 5, shape), rng.integers(0, 5, shape)
        dense = _device(a.astype(np.uint32)).evaluate(_device(b.astype(np.uint32)), size_threshold=3)
        big = _device(ids[a]).evaluate(_device(ids[b]), size_threshold=3)
        assert_scores(big, dense)
        s, g, c = _device(ids[a]).contingency_table(_device(ids[b]))
        ws, wg, wc = O.contingency_pairs(ids[a], ids[b])
        assert np.array_equal(s, ws) and np.array_equal(g, wg) and np.array_equal(c, wc)


@gpu
def test_a_tiny_first_table_grows_to_the_same_result(monkeypatch):
    from chunkflow_b200.chunk import device
    rng = np.random.default_rng(11)
    seg, gt = rng.integers(0, 3000, (20, 40, 40)), rng.integers(0, 700, (20, 40, 40))
    want = _device(seg.astype(np.uint32)).evaluate(_device(gt.astype(np.uint32)), size_threshold=1)
    want_table = _device(seg.astype(np.uint32)).contingency_table(_device(gt.astype(np.uint32)))
    monkeypatch.setattr(device, "EVALUATE_INITIAL_SLOTS", 4)
    got = _device(seg.astype(np.uint32)).evaluate(_device(gt.astype(np.uint32)), size_threshold=1)
    assert_scores(got, want)
    assert_scores(got, O.evaluate(seg, gt, 1))
    for a, b in zip(_device(seg.astype(np.uint32)).contingency_table(_device(gt.astype(np.uint32))), want_table):
        assert np.array_equal(a, b)


@gpu
def test_two_calls_are_bit_identical():
    rng = np.random.default_rng(13)
    field = rng.random((48, 96, 96))
    seg = (field * 40).astype(np.uint32)
    gt = (field * 37 + rng.random(field.shape)).astype(np.uint64)
    s, g = _device(seg), _device(gt)
    a, b = s.evaluate(g), s.evaluate(g)
    for k in O.SCORE_KEYS:
        assert np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes(), k


def _blobs(shape, threshold, seed):
    """Connected components of a smooth thresholded field (labels numbered in raster order)."""
    import torch
    from chunkflow_b200.chunk.device import DeviceChunk
    g = torch.Generator(device="cuda").manual_seed(seed)
    f = torch.randn((1, 1) + shape, device="cuda", generator=g)
    k = torch.ones((1, 1, 5, 5, 5), device="cuda") / 125
    for _ in range(3):
        f = torch.nn.functional.conv3d(f, k, padding=2)
    f = (f[0, 0] / f.std()).contiguous()
    return DeviceChunk(f).connected_component(threshold=threshold)


@gpu
@pytest.mark.slow
def test_large_volume_against_the_oracle():
    """128 x 512 x 512: the sums pass 2^53, where the reference's float64 sums round; rtol 1e-12."""
    seg = _blobs((128, 512, 512), 0.2, 1)
    gt = _blobs((128, 512, 512), 0.6, 2)
    got = seg.evaluate(gt)
    want = O.evaluate(seg.tensor.cpu().numpy().view(np.uint32), gt.tensor.cpu().numpy().view(np.uint32))
    assert_scores(got, want, rtol=1e-12)


@gpu
def test_cli_chain_puts_the_scores_in_the_task(tmp_path):
    from chunkflow_b200.flow import cli
    from chunkflow_b200.chunk.base import Chunk
    gt = np.zeros((16, 64, 64), np.uint32)
    gt[:, :32] = 1
    gt[:, 32:, 10:] = 2
    path = tmp_path / "gt.npy"
    np.save(path, gt)
    tasks = cli.main.main(["create-chunk", "--size", "16", "64", "64", "--dtype", "float32", "to-device",
                           "connected-components", "--threshold", "0.5", "load-npy", "-f", str(path), "-o", "groundtruth",
                           "evaluate-segmentation"], standalone_mode=False)
    seg = Chunk.create(size=(16, 64, 64), dtype=np.float32)
    from oracle import segmentation_oracle as SO
    want = O.evaluate(SO.connected_components(seg.array > 0.5, 6), gt)
    assert_scores(tasks[0]["seg_score"], want)
