"""`agglomerate` (SURVEY.md section 8 f4; reference plugins/agglomerate.py:8-48 -> waterz.agglomerate).

waterz is absent from the reference tree and from this image: the oracle restates its published algorithm ("parity unpinned",
oracle/agglomeration_oracle.py).  On the CPU: the oracle against its own statement-by-statement form of the sequential
watershed, the device code of csrc/watershed_kernels.cuh compiled for the host behind a one-thread CUDA shim
(tests/host_emulation/ws_emulation.cpp) against the oracle, and the native library's host merge loop against the oracle.
On the GPU: the CUDA kernels through the C ABI against the oracle, plus size-independent properties on a larger volume."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import agglomeration_oracle as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOW, HIGH = 0.001, 0.9999


def _affinities(seed, shape, kind):
    """kind: 0 random float32 (no ties), 1 quantised to quarters (plateaus), 2 a saturated block (>= HIGH), 3 zeros below 0.3
    (background), 4 NaNs sprinkled in, 5 smooth (neighbouring voxels alike, like a network output)."""
    rng = np.random.default_rng(seed)
    a = rng.random((3,) + tuple(shape)).astype(np.float32)
    if kind == 1:
        a = (np.round(a * 4) / 4 * 0.9).astype(np.float32)
    elif kind == 2:
        a[:, : shape[0] // 2 + 1, : shape[1] // 2 + 1] = 1.0
    elif kind == 3:
        a[a < 0.3] = 0.0
    elif kind == 4:
        a[rng.random(a.shape) < 0.05] = np.nan
    elif kind == 5:
        from scipy import ndimage
        a = ndimage.gaussian_filter(rng.standard_normal(a.shape), sigma=(0, 1.0, 2.0, 2.0))
        a = (1.0 / (1.0 + np.exp(-4.0 * a / a.std()))).astype(np.float32)
    return a


# ------------------------------------------------------------------------------------------------------------
# oracle self-consistency
# ------------------------------------------------------------------------------------------------------------
def test_oracle_watershed_known_answers():
    # one row of four voxels, x affinities 0.9 | 0.2 | 0.8: two basins split at the weak edge
    a = np.zeros((3, 1, 1, 4), np.float32)
    a[2, 0, 0, 1:] = (0.9, 0.2, 0.8)
    assert A.watershed(a, LOW, HIGH).tolist() == [[[1, 1, 2, 2]]]
    assert A.watershed_literal(a, LOW, HIGH).tolist() == [[[1, 1, 2, 2]]]
    # nothing exceeds the low threshold: all background; everything saturated: one fragment
    assert not A.watershed(np.zeros((3, 2, 3, 3), np.float32), LOW, HIGH).any()
    assert (A.watershed(np.ones((3, 2, 3, 3), np.float32), LOW, HIGH) == 1).all()
    # region graph + scores of the row: fragments 1 | 2 share one face with affinity 0.2
    u, v, s, c = A.region_graph(a, np.array([[[1, 1, 2, 2]]]))
    assert (u.tolist(), v.tolist(), c.tolist()) == ([1], [2], [1]) and s[0] == int(np.rint(np.float64(np.float32(0.2)) * 2 ** 30))
    assert A.agglomerate_edges(3, u, v, s, c, 0.7).tolist() == [0, 1, 2]      # score 0.8 >= 0.7: no merge
    assert A.agglomerate_edges(3, u, v, s, c, 0.85).tolist() == [0, 1, 1]     # merged, the smaller id survives
    # the plugin flips chunkflow's x, y, z channel order before anything else (reference agglomerate.py:26-29)
    assert A.agglomerate(a[::-1], 0.85).tolist() == [[[1, 1, 1, 1]]] and A.agglomerate(a[::-1], 0.7).dtype == np.uint64


@pytest.mark.parametrize("kind", [0, 2, 3])
def test_order_independent_watershed_equals_the_sequential_statement(kind):
    """Without exact ties below the high threshold no plateau has an interior, and the form the kernels implement is the
    sequential algorithm's result, ids included."""
    for seed, shape in ((0, (5, 7, 9)), (1, (8, 6, 4)), (2, (1, 9, 11))):
        a = _affinities(seed, shape, kind)
        assert np.array_equal(A.watershed(a, LOW, HIGH), A.watershed_literal(a, LOW, HIGH)), (kind, seed)


def test_plateau_interiors_are_where_the_two_forms_may_differ():
    """Coarsely quantised maps have plateaus with interior voxels; the two forms still agree on the foreground and on most
    basins (documented deviation: queue order inside a breadth-first level is not reproduced)."""
    same = total = 0
    for seed in range(8):
        a = _affinities(seed, (6, 12, 14), 1)
        w, l = A.watershed(a, LOW, HIGH), A.watershed_literal(a, LOW, HIGH)
        assert np.array_equal(w > 0, l > 0)
        total += 1
        same += np.array_equal(w, l)
    assert same >= total // 2


# ------------------------------------------------------------------------------------------------------------
# the device code on the host (one-thread CUDA shim)
# ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("ws_emu") / "libws_emu.so"
    src = os.path.join(ROOT, "tests", "host_emulation", "ws_emulation.cpp")
    subprocess.run([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", src, "-o", str(out)], check=True)
    lib = C.CDLL(str(out))
    lib.emu_region_graph.restype = C.c_int64
    return lib


def _p(a):
    return C.c_void_p(a.ctypes.data)


def _emu_watershed(lib, affs, flip):
    affs = np.ascontiguousarray(affs, np.float32)
    z, y, x = affs.shape[1:]
    out = np.empty((z, y, x), np.uint32)
    n = lib.emu_watershed(_p(affs), C.c_int(flip), C.c_int64(z), C.c_int64(y), C.c_int64(x), C.c_float(LOW), C.c_float(HIGH), _p(out))
    return out, n


def _emu_region_graph(lib, affs, flip, frag, slots):
    affs, frag = np.ascontiguousarray(affs, np.float32), np.ascontiguousarray(frag, np.uint32)
    z, y, x = frag.shape
    u, v = np.empty(slots, np.uint32), np.empty(slots, np.uint32)
    s, c = np.empty(slots, np.uint64), np.empty(slots, np.uint32)
    n = lib.emu_region_graph(_p(affs), C.c_int(flip), _p(frag), C.c_int64(z), C.c_int64(y), C.c_int64(x), C.c_int64(slots),
                             _p(u), _p(v), _p(s), _p(c))
    k = max(int(n), 0)
    return n, u[:k], v[:k], s[:k], c[:k]


def test_kernel_logic_on_the_host_against_the_oracle(emu):
    rng = np.random.default_rng(42)
    for trial in range(24):
        shape = tuple(int(v) for v in rng.integers(1, 12, 3))
        a = _affinities(100 + trial, shape, trial % 5)
        ref = A.watershed(a, LOW, HIGH)
        got, n = _emu_watershed(emu, a, 0)
        assert n == ref.max() and np.array_equal(got, ref), (trial, shape)
        got_flipped, _ = _emu_watershed(emu, a[::-1], 1)          # chunkflow's channel order, read in reverse
        assert np.array_equal(got_flipped, ref), (trial, shape)
        u, v, s, c = A.region_graph(a, ref)
        slots = 1 << max(4, int(np.ceil(np.log2(2 * len(u) + 1))))
        n, gu, gv, gs, gc = _emu_region_graph(emu, a, 0, ref, slots)
        assert n == len(u) and np.array_equal(gu, u) and np.array_equal(gv, v) and np.array_equal(gs, s) and np.array_equal(gc, c)
        if len(u) > 2:
            assert _emu_region_graph(emu, a, 0, ref, 2)[0] == -1   # a table that cannot hold the pairs reports it


def test_whole_operator_with_emulated_voxel_passes_and_the_native_merge_loop(emu):
    """fragments (emulated kernels) -> region graph (emulated kernels) -> cfb_agglomerate_edges_host (the product's host code)
    -> relabel (emulated kernel) == the oracle's plugin."""
    from chunkflow_b200 import _native
    for seed, shape, kind, thr in ((0, (6, 10, 12), 0, 0.5), (1, (8, 12, 12), 5, 0.3), (2, (5, 9, 9), 1, 0.8), (3, (4, 8, 8), 2, 0.2)):
        a = _affinities(seed, shape, kind)              # stored in chunkflow's order x, y, z
        frag, n = _emu_watershed(emu, a, 1)
        cnt, u, v, s, c = _emu_region_graph(emu, a, 1, frag, 1 << 14)
        root = _native.agglomerate_edges_host(n + 1, u, v, s, c, thr)
        seg = np.empty_like(frag)
        emu.emu_relabel(_p(frag), C.c_int64(frag.size), _p(root), C.c_uint32(root.size), _p(seg))
        assert np.array_equal(seg.astype(np.uint64), A.agglomerate(a, thr, flip_channel=True)), (seed, kind)


# ------------------------------------------------------------------------------------------------------------
# the host merge loop of the native library (no GPU involved)
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,threads,grain", [("0", "1", "2048"), ("1", "1", "2048"), ("1", "6", "500"), ("2", "3", "64")])
def test_native_merge_loop_against_the_oracle(monkeypatch, mode, threads, grain):
    from chunkflow_b200 import _native
    monkeypatch.setenv("CFB_AGGLOMERATE_MODE", mode)
    monkeypatch.setenv("CFB_AGGLOMERATE_THREADS", threads)
    monkeypatch.setenv("CFB_AGGLOMERATE_GRAIN", grain)
    rng = np.random.default_rng(7)
    # (the last two graphs have more than 4096 edges: in mode 1 they go through rounds, pruning and the hand-over to the walk)
    for trial, (shape, thr, kind) in enumerate((((6, 10, 12), 0.5, 0), ((8, 12, 12), 0.3, 5), ((5, 9, 9), 0.8, 1), ((10, 16, 16), 0.45, 0),
                                                ((12, 28, 28), 0.5, 0), ((10, 30, 30), 0.35, 5))):
        a = _affinities(trial, shape, kind)
        frag = A.watershed(a, LOW, HIGH)
        u, v, s, c = A.region_graph(a, frag)
        n = int(frag.max()) + 1
        assert np.array_equal(_native.agglomerate_edges_host(n, u, v, s, c, thr), A.agglomerate_edges(n, u, v, s, c, thr))
    # a random sparse graph with MANY equal scores: the tie rule (score, smaller id, larger id) decides
    n = 1500
    pairs = set()
    while len(pairs) < 6000:
        p, q = (int(t) for t in rng.integers(1, n, 2))
        if p != q:
            pairs.add((min(p, q), max(p, q)))
    pairs = sorted(pairs)
    u = np.array([p for p, _ in pairs], np.uint32)
    v = np.array([q for _, q in pairs], np.uint32)
    c = rng.integers(1, 5, len(u)).astype(np.uint32)
    s = (rng.integers(0, 5, len(u)) * c.astype(np.int64) * (1 << 28)).astype(np.uint64)
    for thr in (0.2, 0.5, 0.76, 1.5):
        ref = A.agglomerate_edges(n, u, v, s, c, thr)
        assert np.array_equal(_native.agglomerate_edges_host(n, u, v, s, c, thr), ref)
        assert np.array_equal(ref[ref], ref) and (ref <= np.arange(n)).all()    # idempotent; the smallest id of a cluster survives
    assert _native.agglomerate_edges_host(3, [], [], [], [], 0.5).tolist() == [0, 1, 2]
    with pytest.raises(_native.NativeError):
        _native.agglomerate_edges_host(3, [1], [5], [1], [1], 0.5)       # id outside the node range
    with pytest.raises(_native.NativeError):
        _native.agglomerate_edges_host(3, [1, 1], [2, 2], [1, 1], [1, 1], 0.5)   # duplicate edge


@pytest.mark.parametrize("mode,threads,grain", [("0", "1", "2048"), ("1", "4", "2048"), ("2", "1", "2048"), ("2", "5", "3"), ("2", "8", "1")])
def test_native_merge_loop_fuzz_shapes_ties_and_odd_thresholds(monkeypatch, mode, threads, grain):
    """Random, chain, star + ring and dense graphs with few distinct means (ties everywhere), means above 1 (negative scores),
    thresholds 0 / 1 / 2 / negative / inf: the native loop == the oracle's heap walk, in each of its modes -- 0: the sequential
    walk alone (bucket queue, shorter list moved), 2: rounds of mutual-best merges until none is left (on graphs of any size:
    the reducibility argument put to the test, ties included), 1: the product's mix (rounds on large graphs, then the walk);
    the rounds with one worker and with several workers on slices of a few edges each (atomic minima, range-partitioned merge)."""
    from chunkflow_b200 import _native
    monkeypatch.setenv("CFB_AGGLOMERATE_MODE", mode)
    monkeypatch.setenv("CFB_AGGLOMERATE_THREADS", threads)
    monkeypatch.setenv("CFB_AGGLOMERATE_GRAIN", grain)
    rng = np.random.default_rng(123)
    for t in range(160):
        n = int(rng.integers(2, 40))
        kind = t % 4
        pairs = set()
        if kind == 0:
            for _ in range(int(rng.integers(0, n * 3))):
                a, b = (int(x) for x in rng.integers(1, n, 2))
                if a != b:
                    pairs.add((min(a, b), max(a, b)))
        elif kind == 1:
            pairs = {(i, i + 1) for i in range(1, n - 1)}
        elif kind == 2:
            pairs = {(1, i) for i in range(2, n)} | {(i, i + 1) for i in range(2, n - 1)}
        else:
            pairs = {(a, b) for a in range(1, n) for b in range(a + 1, n) if rng.random() < 0.5}
        pairs = sorted(pairs)
        u = np.array([p for p, _ in pairs], np.uint32)
        v = np.array([q for _, q in pairs], np.uint32)
        c = rng.integers(1, 4, len(u)).astype(np.uint32)
        levels = int(rng.choice([2, 3, 5, 1000]))
        mean = rng.integers(0, levels + 1, len(u)) / levels * float(rng.choice([1.0, 1.0, 1.3]))
        s = np.rint(mean * c * (1 << 30)).astype(np.uint64)
        for thr in (float(rng.random()), 0.0, 1.0, 2.0, -0.5, float("inf")):
            assert np.array_equal(_native.agglomerate_edges_host(n, u, v, s, c, thr), A.agglomerate_edges(n, u, v, s, c, thr)), (t, thr)


def test_threaded_rounds_under_thread_sanitizer(tmp_path):
    """The worker threads of the rounds share arrays through relaxed atomics and disjoint slices: ThreadSanitizer must stay
    silent, and eight workers must return what one worker returns."""
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    exe = tmp_path / "tsan_agglomerate"
    cmd = [gxx, "-O1", "-g", "-std=c++17", "-fsanitize=thread", "-x", "c++", "-I/usr/local/cuda/include",
           "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "chunkflow_b200", "csrc"),
           os.path.join(ROOT, "chunkflow_b200", "csrc", "agglomerate_host.cu"),
           os.path.join(ROOT, "tests", "host_emulation", "tsan_agglomerate.cpp"), "-o", str(exe), "-lpthread"]
    build = subprocess.run(cmd, capture_output=True, text=True)
    if build.returncode != 0:
        pytest.skip("no ThreadSanitizer build here: " + build.stderr[-300:])
    run = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    if "unexpected memory mapping" in run.stderr or "FATAL: ThreadSanitizer" in run.stderr:
        pytest.skip("ThreadSanitizer cannot run in this sandbox")
    assert run.returncode == 0 and "bad 0" in run.stdout, run.stdout[-500:] + run.stderr[-2000:]
    assert "WARNING: ThreadSanitizer" not in run.stderr, run.stderr[-3000:]


def test_plugin_refuses_other_scoring_functions_and_needs_a_gpu():
    from chunkflow_b200 import Chunk
    from chunkflow_b200.plugins import agglomerate
    affs = Chunk(np.zeros((3, 2, 4, 4), np.float32))
    with pytest.raises(NotImplementedError):
        agglomerate.execute(affs, scoring_function='OneMinus<MaxAffinity<RegionGraphType, ScoreValue>>')
    from conftest import has_gpu
    if not has_gpu():
        with pytest.raises(Exception):       # no CPU fallback
            agglomerate.execute(affs)


def test_plugin_signature_matches_the_reference_plugin(pins):
    """Same parameter names, order and defaults as chunkflow/plugins/agglomerate.py: execute (read with `ast` by
    tests/golden/make_golden_reference.py: importing the reference module needs waterz), plus the trailing `device`
    extension; the CLI command carries the same knobs."""
    import inspect
    from chunkflow_b200.flow import cli
    from chunkflow_b200.plugins import agglomerate
    from reference_pins import REQUIRED, plain
    ours = inspect.signature(agglomerate.execute)
    expected = [("affs", inspect.Parameter.empty), ("fragments", None), ("threshold", 0.7), ("aff_threshold_low", 0.001),
                ("aff_threshold_high", 0.9999), ("scoring_function", 'OneMinus<MeanAffinity<RegionGraphType, ScoreValue>>'),
                ("flip_channel", True)]
    assert plain([[n, REQUIRED if d is inspect.Parameter.empty else d] for n, d in expected]) == \
        pins.get("agglomerate/execute_signature")
    got = [(n, p.default) for n, p in ours.parameters.items()]
    assert got[:len(expected)] == expected and [n for n, _ in got[len(expected):]] == ["device"]
    opts = {o for p in cli.agglomerate.params for o in p.opts + p.secondary_opts}
    for flag in ("--threshold", "--aff-threshold-low", "--aff-threshold-high", "--flip-channel", "--no-flip-channel",
                 "--input-chunk-name", "--output-chunk-name", "--name"):
        assert flag in opts, flag
    assert {p.name: p.default for p in cli.agglomerate.params}["threshold"] == 0.7


# ------------------------------------------------------------------------------------------------------------
# GPU: the CUDA kernels through the C ABI
# ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_watershed_and_region_graph_against_the_oracle():
    import torch
    from chunkflow_b200 import _native
    from chunkflow_b200.chunk.device import DeviceChunk
    cases = [(0, (17, 40, 53), 0), (1, (9, 33, 64), 1), (2, (12, 30, 31), 2), (3, (8, 20, 20), 3), (4, (6, 25, 17), 4), (5, (24, 48, 48), 5),
             (6, (1, 1, 7), 0), (7, (1, 16, 16), 1), (8, (33, 5, 3), 0)]
    for seed, shape, kind in cases:
        a = _affinities(seed, shape, kind)                      # waterz order z, y, x
        ref = A.watershed(a, LOW, HIGH)
        for flip in (False, True):
            stored = np.ascontiguousarray(a[::-1]) if flip else a
            dev = DeviceChunk(torch.from_numpy(stored).cuda(), voxel_offset=(1, 2, 3), voxel_size=(4, 4, 4), layer_type="affinity_map")
            frag = dev.watershed(LOW, HIGH, flip_channel=flip)
            got = frag.tensor.cpu().numpy().view(np.uint32)
            assert frag.num_components == ref.max() and tuple(frag.voxel_offset) == (1, 2, 3)
            assert np.array_equal(got, ref), (seed, kind, flip)
            u, v, s, c = dev.region_graph(frag, flip_channel=flip)
            ru, rv, rs, rc = A.region_graph(a, ref)
            assert np.array_equal(u, ru) and np.array_equal(v, rv) and np.array_equal(s, rs) and np.array_equal(c, rc), (seed, kind, flip)
    # a table that is too small is reported, not overrun
    a = _affinities(0, (17, 40, 53), 0)
    dev = DeviceChunk(torch.from_numpy(a).cuda(), layer_type="affinity_map")
    frag = dev.watershed(LOW, HIGH, flip_channel=False)
    work = torch.empty(_native.region_graph_workspace(16), dtype=torch.uint8, device="cuda")
    with pytest.raises(_native.NativeError) as err:
        _native.region_graph_device(dev.tensor.data_ptr(), False, frag.tensor.data_ptr(), frag.shape, work.data_ptr(), 16)
    assert err.value.code == _native.ERR_CAPACITY


@pytest.mark.gpu
def test_device_agglomerate_plugin_and_cli_against_the_oracle():
    import torch
    from click.testing import CliRunner
    from chunkflow_b200 import Chunk
    from chunkflow_b200.chunk.device import DeviceChunk
    from chunkflow_b200.flow import cli
    from chunkflow_b200.plugins import agglomerate
    for seed, shape, kind, thr in ((0, (12, 30, 31), 5, 0.3), (1, (9, 20, 24), 0, 0.5), (2, (6, 16, 16), 1, 0.8), (3, (8, 20, 20), 2, 0.2),
                                   (4, (10, 24, 24), 3, 0.6)):
        a = _affinities(seed, shape, kind)                      # chunkflow's order x, y, z: the plugin flips
        ref = A.agglomerate(a, thr, aff_threshold_low=LOW, aff_threshold_high=HIGH)
        out = agglomerate.execute(Chunk(a, voxel_offset=(5, 6, 7), voxel_size=(40, 4, 4)), threshold=thr, aff_threshold_low=LOW,
                                  aff_threshold_high=HIGH)
        assert isinstance(out, list) and len(out) == 1
        seg = out[0]
        assert seg.array.dtype == np.uint64 and tuple(seg.voxel_offset) == (5, 6, 7)
        assert np.array_equal(seg.array, ref), (seed, kind)
        # fragments handed in (here: connected components of the thresholded mean affinity) instead of the watershed
        frag = A.watershed(np.flip(a, 0), 0.3, 0.8)
        ref2 = A.agglomerate(a, thr, fragments=frag)
        out2 = agglomerate.execute(Chunk(a), fragments=frag.astype(np.uint64), threshold=thr)[0]
        assert np.array_equal(out2.array, ref2), (seed, kind)
    # DeviceChunk API keeps everything on the GPU; threshold 0 merges nothing
    a = _affinities(9, (10, 24, 24), 5)
    dev = DeviceChunk(torch.from_numpy(a).cuda(), layer_type="affinity_map")
    seg0 = dev.agglomerate(threshold=0.0)
    assert np.array_equal(seg0.tensor.cpu().numpy().view(np.uint32), A.watershed(np.flip(a, 0), LOW, HIGH))
    assert seg0.num_components == seg0.num_fragments
    # CLI, the README pipeline (reference README.md:39): inference -> agglomerate; the identity backend turns the image into
    # a 3-channel map in [0, 1] (full of exact ties: plateaus everywhere)
    pipeline = ["create-chunk", "--size", "16", "64", "64", "--pattern", "sin",
                "inference", "--input-patch-size", "8", "32", "32", "--output-patch-overlap", "2", "8", "8",
                "--num-output-channels", "3", "--framework", "identity", "--batch-size", "4", "--mask-output-chunk"]
    res = CliRunner().invoke(cli.main, pipeline + ["agglomerate", "--threshold", "0.4", "-o", "seg"], standalone_mode=False)
    assert res.exception is None, res.output
    task = res.return_value[0]
    assert "agglomerate" in task["log"]["timer"]
    # the oracle works on the affinity map of THIS task (the blend's float atomics differ in the last bit from run to run,
    # and on a map full of ties that moves watershed boundaries)
    affs = np.asarray(task["chunk"].array)
    assert affs.shape == (3, 16, 64, 64)
    assert np.array_equal(np.asarray(task["seg"].array).astype(np.uint64), A.agglomerate(affs, 0.4))


@pytest.mark.gpu
def test_agglomerate_properties_on_a_larger_volume():
    """Size-independent properties where the pure-Python oracle would take minutes: gapless fragment ids, background exactly
    where no affinity exceeds the low threshold, the region graph's face count, surviving ids = smallest id of each cluster,
    coarser thresholds only merge."""
    import torch
    from chunkflow_b200.chunk.device import DeviceChunk
    a = _affinities(11, (48, 192, 192), 5)
    a[:, :4] = 0.0                                          # a slab without affinities: background
    dev = DeviceChunk(torch.from_numpy(a).cuda(), layer_type="affinity_map")
    frag = dev.watershed(LOW, HIGH)
    f = frag.tensor.cpu().numpy().view(np.uint32)
    n = frag.num_components
    assert f.max() == n and np.array_equal(np.unique(f), np.arange(0, n + 1))
    w = A._edge_weights(np.ascontiguousarray(a[::-1]), LOW)
    assert np.array_equal(f == 0, ~(w.max(axis=0) > np.float32(LOW)))
    first = np.unique(f.ravel(), return_index=True)[1][1:]
    assert np.all(np.diff(first) > 0)                       # ids in raster order of the first voxel
    u, v, s, c = dev.region_graph(frag)
    ru, rv, rs, rc = A.region_graph(np.ascontiguousarray(a[::-1]), f)     # (numpy: vectorised, fast enough)
    assert np.array_equal(u, ru) and np.array_equal(v, rv) and np.array_equal(s, rs) and np.array_equal(c, rc)
    lo = dev.agglomerate(threshold=0.3, fragments=frag).tensor.cpu().numpy().view(np.uint32)
    hi = dev.agglomerate(threshold=0.6, fragments=frag).tensor.cpu().numpy().view(np.uint32)
    for seg in (lo, hi):
        assert np.array_equal(seg == 0, f == 0) and (seg <= f).all()
        pairs = np.unique(np.stack([f.ravel(), seg.ravel()]), axis=1)
        assert len(pairs[0]) == n + 1                       # every fragment goes to exactly one segment
        assert np.array_equal(np.unique(seg), np.unique(pairs[1]))
        mins = {}
        for fr, sg in zip(pairs[0].tolist(), pairs[1].tolist()):
            mins[sg] = min(mins.get(sg, fr), fr)
        assert all(k == m for k, m in mins.items())         # the surviving id is the smallest fragment id of the cluster
    assert len(np.unique(hi)) <= len(np.unique(lo)) <= n + 1
