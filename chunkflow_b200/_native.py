"""ctypes binding of ``include/chunkflow_b200.h`` (the C-ABI of the CUDA hot path).

The library is loaded lazily and LOUDLY: if ``libchunkflow_b200.so`` is missing (and
cannot be built) or no CUDA device is present, every compute entry point raises --
there is no CPU fallback in the product path.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

OK = 0
ERR_INVALID_ARGUMENT, ERR_CUDA, ERR_WEIGHTS, ERR_OUTPUT_RANGE, ERR_UNSUPPORTED, ERR_CAPACITY = -1, -2, -3, -4, -5, -6
FRAMEWORK_UNET3L, FRAMEWORK_IDENTITY = 0, 1
PRECISION_F32_SIMT, PRECISION_F16X3_UMMA, PRECISION_F16_UMMA, PRECISION_F16F8_UMMA = 0, 1, 2, 3
DTYPE_U8, DTYPE_F32, DTYPE_U32, DTYPE_U64 = 0, 1, 2, 3
AUGMENT_NONE, AUGMENT_REFERENCE, AUGMENT_SPATIAL = 0, 1, 2
QUANTIZE_XY, QUANTIZE_Z = 0, 1

# every symbol include/chunkflow_b200.h declares
EXPORTS = (
    "cfb_last_error", "cfb_version", "cfb_device_count", "cfb_device_memory", "cfb_create", "cfb_destroy", "cfb_device_name",
    "cfb_set_weight", "cfb_commit_weights", "cfb_patch_mask", "cfb_patch_grid", "cfb_output_shape",
    "cfb_infer_chunk_device", "cfb_infer_chunk_host", "cfb_infer_slab_device", "cfb_normalize_device",
    "cfb_slab_nonzero", "cfb_halo_add_device", "cfb_weight_volume_device",
    "cfb_patch_forward_host", "cfb_make_patch_mask", "cfb_plugin_begin", "cfb_plugin_extract", "cfb_plugin_blend",
    "cfb_plugin_end", "cfb_last_timing", "cfb_set_profiling", "cfb_layer_timing", "cfb_debug_net_forward_host", "cfb_debug_conv3_host",
    "cfb_normalize_contrast_device", "cfb_maskout_device", "cfb_crop_margin_device", "cfb_quantize_device",
    "cfb_connected_components_device", "cfb_connected_components_workspace",
    "cfb_watershed_workspace", "cfb_watershed_device", "cfb_region_graph_workspace", "cfb_region_graph_device",
    "cfb_region_graph_read", "cfb_agglomerate_edges_host", "cfb_relabel_device",
    "cfb_contingency_workspace", "cfb_contingency_device", "cfb_contingency_scores", "cfb_contingency_read",
)


class Params(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("device", C.c_int32), ("framework", C.c_int32), ("precision", C.c_int32),
        ("input_patch_size", C.c_int32 * 3), ("output_patch_size", C.c_int32 * 3),
        ("output_patch_overlap", C.c_int32 * 3), ("output_crop_margin", C.c_int32 * 3),
        ("num_input_channels", C.c_int32), ("num_output_channels", C.c_int32), ("batch_size", C.c_int32),
        ("mask_output_chunk", C.c_int32), ("augment", C.c_int32), ("has_myelin_threshold", C.c_int32),
        ("mask_myelin_threshold", C.c_float), ("check_output_range", C.c_int32),
    ]


class ContingencySums(C.Structure):
    """cfb_contingency_sums (include/chunkflow_b200.h)."""
    _fields_ = [(n, C.c_uint64) for n in ("voxels", "entries", "sum_sq_pairs", "sum_sq_seg", "sum_sq_gt", "nonzero_voxels",
                                          "seg_labels", "pairs_over_threshold")] + \
               [(n, C.c_uint64 * 2) for n in ("xlogx_pairs", "xlogx_seg", "xlogx_gt")]


class NativeError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"chunkflow_b200 native error {code}: {message}")
        self.code = code


_lib: Optional[C.CDLL] = None


def library_path() -> str:
    from .build import LIB_PATH
    return LIB_PATH


def load() -> C.CDLL:
    """Load (building in-tree first if the sources are newer) the native library."""
    global _lib
    if _lib is not None:
        return _lib
    from .build import build_native, LIB_PATH
    path = LIB_PATH
    override = os.environ.get("CFB_NATIVE_LIB")  # development: an instrumented build (python -m chunkflow_b200.build --variant)
    try:
        path = override if override else build_native()
        if override and not os.path.exists(override):
            raise RuntimeError(f"CFB_NATIVE_LIB={override} does not exist")
    except Exception as exc:  # no nvcc on this box: use the prebuilt .so that travelled with the tree
        if override or not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "chunkflow_b200: the CUDA extension libchunkflow_b200.so is missing and could not be built "
                f"({exc}); there is no CPU fallback") from exc
    lib = C.CDLL(path)
    vp, i32, i64, f32p = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_float)
    lib.cfb_last_error.restype = C.c_char_p
    lib.cfb_device_name.restype = C.c_char_p
    lib.cfb_device_name.argtypes = [vp]
    lib.cfb_version.restype = C.c_int
    lib.cfb_device_count.restype = C.c_int
    lib.cfb_device_memory.argtypes = [i32, C.POINTER(i64), C.POINTER(i64)]
    lib.cfb_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    lib.cfb_destroy.argtypes = [vp]
    lib.cfb_set_weight.argtypes = [vp, C.c_char_p, vp, i64]
    lib.cfb_commit_weights.argtypes = [vp]
    lib.cfb_patch_mask.argtypes = [vp, vp]
    lib.cfb_patch_grid.argtypes = [vp, i64, i64, i64, C.POINTER(i64), vp, i64]
    lib.cfb_output_shape.argtypes = [vp, i64, i64, i64, C.POINTER(i64 * 4)]
    lib.cfb_infer_chunk_device.argtypes = [vp, vp, i32, i64, i64, i64, vp, vp]
    lib.cfb_infer_chunk_host.argtypes = [vp, vp, i32, i64, i64, i64, vp]
    lib.cfb_infer_slab_device.argtypes = [vp, vp, i32, i64, i64, i64, i64, i64, vp, vp, vp]
    lib.cfb_normalize_device.argtypes = [vp, vp, vp, i32, i64, i64, i64, i64, i32, vp]
    lib.cfb_slab_nonzero.argtypes = [vp, C.POINTER(i32), vp]
    lib.cfb_halo_add_device.argtypes = [vp, vp, i64, vp]
    lib.cfb_weight_volume_device.argtypes = [vp, i64, i64, i64, i64, i64, i32, vp, vp]
    lib.cfb_patch_forward_host.argtypes = [vp, vp, i32, vp]
    lib.cfb_make_patch_mask.argtypes = [C.POINTER(i32 * 3), C.POINTER(i32 * 3), vp]
    lib.cfb_plugin_begin.argtypes = [vp, vp, i32, i64, i64, i64]
    lib.cfb_plugin_extract.argtypes = [vp, i64, i32, vp]
    lib.cfb_plugin_blend.argtypes = [vp, i64, i32, vp]
    lib.cfb_plugin_end.argtypes = [vp, vp]
    lib.cfb_last_timing.argtypes = [vp, C.POINTER(C.c_float * 5), C.POINTER(i64)]
    lib.cfb_set_profiling.argtypes = [vp, i32]
    lib.cfb_layer_timing.argtypes = [vp, i32, C.POINTER(i32), vp, vp, vp]
    lib.cfb_debug_net_forward_host.argtypes = [vp, vp, vp]
    lib.cfb_debug_conv3_host.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, i32, i32, vp]
    lib.cfb_normalize_contrast_device.argtypes = [vp, i64, i64, i64, C.c_double, C.c_double, i32, i32, i32, vp]
    lib.cfb_maskout_device.argtypes = [vp, i32, i64, i64, i64, i64, vp, i32, i64, i64, i64, vp]
    lib.cfb_crop_margin_device.argtypes = [vp, i32, i64, i64, i64, i64, C.POINTER(i64 * 6), vp, vp]
    lib.cfb_quantize_device.argtypes = [vp, i64, i64, i64, i64, i32, vp, vp]
    lib.cfb_connected_components_device.argtypes = [vp, i32, i64, i64, i64, C.c_float, i32, vp, vp, C.POINTER(C.c_uint32), vp]
    lib.cfb_connected_components_workspace.argtypes = [i64, i64, i64]
    lib.cfb_connected_components_workspace.restype = i64
    lib.cfb_watershed_workspace.argtypes = [i64, i64, i64]
    lib.cfb_watershed_workspace.restype = i64
    lib.cfb_watershed_device.argtypes = [vp, i32, i64, i64, i64, C.c_float, C.c_float, vp, vp, C.POINTER(C.c_uint32), vp]
    lib.cfb_region_graph_workspace.argtypes = [i64]
    lib.cfb_region_graph_workspace.restype = i64
    lib.cfb_region_graph_device.argtypes = [vp, i32, vp, i64, i64, i64, vp, i64, C.POINTER(i64), vp]
    lib.cfb_region_graph_read.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp]
    lib.cfb_agglomerate_edges_host.argtypes = [i64, i64, vp, vp, vp, vp, C.c_float, vp]
    lib.cfb_relabel_device.argtypes = [vp, i64, vp, i64, vp, vp]
    lib.cfb_contingency_workspace.argtypes = [i64]
    lib.cfb_contingency_workspace.restype = i64
    lib.cfb_contingency_device.argtypes = [vp, i32, vp, i32, i64, vp, i64, C.POINTER(i64), vp]
    lib.cfb_contingency_scores.argtypes = [vp, i64, i64, i64, C.c_double, C.POINTER(ContingencySums), vp]
    lib.cfb_contingency_read.argtypes = [vp, i64, i64, vp, vp, vp, vp]
    for name in EXPORTS:
        getattr(lib, name)   # every declared symbol must be there
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != OK:
        raise NativeError(code, load().cfb_last_error().decode("utf-8", "replace"))


def _ptr(a: np.ndarray) -> C.c_void_p:
    return C.c_void_p(a.ctypes.data)


# ---- operators either side of `inference` on device pointers (include/chunkflow_b200.h, SURVEY section 8 f3) ----
def normalize_contrast_device(d_image: int, zyx, lower_clip_fraction: float, upper_clip_fraction: float, minval: int,
                              maxval: int, per_section: bool, stream: int = 0) -> None:
    check(load().cfb_normalize_contrast_device(C.c_void_p(d_image), *(int(v) for v in zyx), float(lower_clip_fraction),
                                               float(upper_clip_fraction), int(minval), int(maxval), int(bool(per_section)),
                                               C.c_void_p(stream)))


def maskout_device(d_chunk: int, chunk_dtype: int, czyx, d_mask: int, mask_dtype: int, factor, stream: int = 0) -> None:
    check(load().cfb_maskout_device(C.c_void_p(d_chunk), int(chunk_dtype), *(int(v) for v in czyx), C.c_void_p(d_mask),
                                    int(mask_dtype), *(int(v) for v in factor), C.c_void_p(stream)))


def crop_margin_device(d_src: int, dtype: int, czyx, margin6, d_dst: int, stream: int = 0) -> None:
    m = (C.c_int64 * 6)(*(int(v) for v in margin6))
    check(load().cfb_crop_margin_device(C.c_void_p(d_src), int(dtype), *(int(v) for v in czyx), C.byref(m), C.c_void_p(d_dst),
                                        C.c_void_p(stream)))


def quantize_device(d_affinity: int, czyx, mode: int, d_out: int, stream: int = 0) -> None:
    check(load().cfb_quantize_device(C.c_void_p(d_affinity), *(int(v) for v in czyx), int(mode), C.c_void_p(d_out),
                                     C.c_void_p(stream)))


def connected_components_workspace(zyx) -> int:
    return int(load().cfb_connected_components_workspace(*(int(v) for v in zyx)))


def connected_components_device(d_in: int, in_dtype: int, zyx, threshold: float, connectivity: int, d_labels: int, d_workspace: int,
                                stream: int = 0) -> int:
    """-> number of components (synchronises the stream)."""
    n = C.c_uint32()
    check(load().cfb_connected_components_device(C.c_void_p(d_in), int(in_dtype), *(int(v) for v in zyx), float(threshold or 0.0),
                                                 int(connectivity), C.c_void_p(d_labels), C.c_void_p(d_workspace), C.byref(n),
                                                 C.c_void_p(stream)))
    return int(n.value)


# ---- `agglomerate` (include/chunkflow_b200.h, SURVEY section 8 f4) ----
def watershed_workspace(zyx) -> int:
    return int(load().cfb_watershed_workspace(*(int(v) for v in zyx)))


def watershed_device(d_affs: int, flip_channel: bool, zyx, aff_threshold_low: float, aff_threshold_high: float, d_fragments: int,
                     d_workspace: int, stream: int = 0) -> int:
    """-> number of fragments (synchronises the stream)."""
    n = C.c_uint32()
    check(load().cfb_watershed_device(C.c_void_p(d_affs), int(bool(flip_channel)), *(int(v) for v in zyx), float(aff_threshold_low),
                                      float(aff_threshold_high), C.c_void_p(d_fragments), C.c_void_p(d_workspace), C.byref(n),
                                      C.c_void_p(stream)))
    return int(n.value)


def region_graph_workspace(table_slots: int) -> int:
    return int(load().cfb_region_graph_workspace(int(table_slots)))


def region_graph_device(d_affs: int, flip_channel: bool, d_fragments: int, zyx, d_workspace: int, table_slots: int,
                        stream: int = 0) -> int:
    """-> number of edges; raises NativeError with code ERR_CAPACITY when the table is too small."""
    n = C.c_int64()
    check(load().cfb_region_graph_device(C.c_void_p(d_affs), int(bool(flip_channel)), C.c_void_p(d_fragments), *(int(v) for v in zyx),
                                         C.c_void_p(d_workspace), int(table_slots), C.byref(n), C.c_void_p(stream)))
    return int(n.value)


def region_graph_read(d_workspace: int, table_slots: int, num_edges: int, stream: int = 0):
    """-> (u, v, sum_fixed, count) host arrays sorted by (u, v)."""
    u, v = np.empty(num_edges, np.uint32), np.empty(num_edges, np.uint32)
    s, c = np.empty(num_edges, np.uint64), np.empty(num_edges, np.uint32)
    check(load().cfb_region_graph_read(C.c_void_p(d_workspace), int(table_slots), int(num_edges), _ptr(u), _ptr(v), _ptr(s), _ptr(c),
                                       C.c_void_p(stream)))
    return u, v, s, c


def agglomerate_edges_host(num_nodes: int, u, v, sum_fixed, count, threshold: float) -> np.ndarray:
    """The merge loop on the host (no GPU involved) -> root_of (num_nodes,) uint32."""
    u = np.ascontiguousarray(u, np.uint32); v = np.ascontiguousarray(v, np.uint32)
    s = np.ascontiguousarray(sum_fixed, np.uint64); c = np.ascontiguousarray(count, np.uint32)
    if not (u.shape == v.shape == s.shape == c.shape and u.ndim == 1):
        raise ValueError("edge arrays must be one-dimensional and of equal length")
    root = np.empty(int(num_nodes), np.uint32)
    check(load().cfb_agglomerate_edges_host(int(num_nodes), int(u.size), _ptr(u), _ptr(v), _ptr(s), _ptr(c), float(threshold), _ptr(root)))
    return root


def relabel_device(d_labels: int, n: int, d_map: int, map_size: int, d_out: int, stream: int = 0) -> None:
    check(load().cfb_relabel_device(C.c_void_p(d_labels), int(n), C.c_void_p(d_map), int(map_size), C.c_void_p(d_out),
                                    C.c_void_p(stream)))


# ---- `evaluate-segmentation` (include/chunkflow_b200.h) ----
def contingency_workspace(table_slots: int) -> int:
    return int(load().cfb_contingency_workspace(int(table_slots)))


def _check_slots(table_slots: int, d_workspace_bytes: Optional[int]) -> None:
    if table_slots < 2 or table_slots & (table_slots - 1):
        raise ValueError("table_slots must be a power of two")
    if d_workspace_bytes is not None and d_workspace_bytes < contingency_workspace(table_slots):
        raise ValueError(f"the workspace holds {d_workspace_bytes} bytes; {table_slots} slots need {contingency_workspace(table_slots)}")


def contingency_device(d_seg: int, seg_dtype: int, d_gt: int, gt_dtype: int, n: int, d_workspace: int, table_slots: int,
                       workspace_bytes: Optional[int] = None, stream: int = 0) -> int:
    """-> number of (seg id, gt id) pairs; raises NativeError with code ERR_CAPACITY when the table is too small."""
    _check_slots(table_slots, workspace_bytes)
    e = C.c_int64()
    check(load().cfb_contingency_device(C.c_void_p(d_seg), int(seg_dtype), C.c_void_p(d_gt), int(gt_dtype), int(n), C.c_void_p(d_workspace),
                                        int(table_slots), C.byref(e), C.c_void_p(stream)))
    return int(e.value)


def contingency_scores(d_workspace: int, table_slots: int, n: int, num_entries: int, size_threshold: float,
                       workspace_bytes: Optional[int] = None, stream: int = 0) -> ContingencySums:
    _check_slots(table_slots, workspace_bytes)
    out = ContingencySums()
    check(load().cfb_contingency_scores(C.c_void_p(d_workspace), int(table_slots), int(n), int(num_entries), float(size_threshold),
                                        C.byref(out), C.c_void_p(stream)))
    return out


def contingency_read(d_workspace: int, table_slots: int, num_entries: int, workspace_bytes: Optional[int] = None, stream: int = 0):
    """-> (seg_ids, gt_ids, counts) uint64 host arrays sorted by (seg id, gt id)."""
    _check_slots(table_slots, workspace_bytes)
    if not 0 <= num_entries <= table_slots // 2:
        raise ValueError("num_entries does not fit the table")
    s, g, c = (np.empty(int(num_entries), np.uint64) for _ in range(3))
    check(load().cfb_contingency_read(C.c_void_p(d_workspace), int(table_slots), int(num_entries), _ptr(s), _ptr(g), _ptr(c),
                                      C.c_void_p(stream)))
    return s, g, c


def device_memory(device: int = 0) -> tuple:
    """(free, total) bytes of device memory."""
    f, t = C.c_int64(), C.c_int64()
    check(load().cfb_device_memory(int(device), C.byref(f), C.byref(t)))
    return f.value, t.value


def make_patch_mask(patch_size, overlap) -> np.ndarray:
    """fp32 bump/patch mask built by the native library (no GPU needed)."""
    ps = (C.c_int32 * 3)(*[int(v) for v in patch_size])
    ov = (C.c_int32 * 3)(*[int(v) for v in overlap])
    out = np.empty(tuple(int(v) for v in patch_size), np.float32)
    check(load().cfb_make_patch_mask(C.byref(ps), C.byref(ov), _ptr(out)))
    return out


def augment_code(augment) -> int:
    """``augment`` as the Inferencer takes it: falsy -> none; True / 'reference' -> the reference's literal arithmetic
    (transform.py:30-52,147-156); 'spatial' -> the 8 spatial flip / transpose variants (explicit opt-in)."""
    if not augment:
        return AUGMENT_NONE
    if augment is True or augment == "reference" or augment == AUGMENT_REFERENCE:
        return AUGMENT_REFERENCE
    if augment == "spatial" or augment == AUGMENT_SPATIAL:
        return AUGMENT_SPATIAL
    raise ValueError(f"augment must be False, True, 'reference' or 'spatial', not {augment!r}")


def halo_add_device(d_dst: int, d_src: int, count: int, stream: int = 0) -> None:
    """d_dst[i] += d_src[i] for `count` float32 on the current device (multi-GPU halo planes)."""
    check(load().cfb_halo_add_device(C.c_void_p(d_dst), C.c_void_p(d_src), int(count), C.c_void_p(stream)))


class Engine:
    """RAII wrapper of a ``cfb_handle``."""

    def __init__(self, *, input_patch_size, output_patch_size, output_patch_overlap, output_crop_margin,
                 num_input_channels=1, num_output_channels=3, batch_size=1, mask_output_chunk=True,
                 framework=FRAMEWORK_UNET3L, precision=PRECISION_F32_SIMT, device=0, augment=False,
                 mask_myelin_threshold=None, check_output_range=True):
        self._h = C.c_void_p()
        self._lib = load()
        p = Params()
        p.struct_size = C.sizeof(Params)
        p.device, p.framework, p.precision = int(device), int(framework), int(precision)
        p.input_patch_size[:] = [int(v) for v in input_patch_size]
        p.output_patch_size[:] = [int(v) for v in output_patch_size]
        p.output_patch_overlap[:] = [int(v) for v in output_patch_overlap]
        p.output_crop_margin[:] = [int(v) for v in output_crop_margin]
        p.num_input_channels, p.num_output_channels = int(num_input_channels), int(num_output_channels)
        p.batch_size, p.mask_output_chunk = int(batch_size), int(bool(mask_output_chunk))
        p.augment = augment_code(augment)
        # truthiness, like the reference (inferencer.py:468: `if self.mask_myelin_threshold:`): None and 0.0 both mean "off"
        p.has_myelin_threshold = int(bool(mask_myelin_threshold))
        p.mask_myelin_threshold = float(mask_myelin_threshold or 0.0)
        p.check_output_range = int(bool(check_output_range))
        self.params = p
        self.input_patch_size = tuple(p.input_patch_size)
        self.output_patch_size = tuple(p.output_patch_size)
        self.num_output_channels = p.num_output_channels
        check(self._lib.cfb_create(C.byref(p), C.byref(self._h)))

    def close(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self._lib.cfb_destroy(h)
            finally:
                self._h = None  # (the ctypes module may already be torn down at interpreter exit)

    __del__ = close

    @property
    def device_name(self) -> str:
        return self._lib.cfb_device_name(self._h).decode()

    def load_state_dict(self, state: dict) -> None:
        for name, tensor in state.items():
            a = np.ascontiguousarray(np.asarray(tensor, dtype=np.float32))
            check(self._lib.cfb_set_weight(self._h, name.encode(), _ptr(a), a.size))
        check(self._lib.cfb_commit_weights(self._h))

    def patch_mask(self) -> np.ndarray:
        out = np.empty(self.output_patch_size, np.float32)
        check(self._lib.cfb_patch_mask(self._h, _ptr(out)))
        return out

    def patch_grid(self, chunk_zyx) -> np.ndarray:
        n = C.c_int64()
        cz, cy, cx = (int(v) for v in chunk_zyx)
        check(self._lib.cfb_patch_grid(self._h, cz, cy, cx, C.byref(n), None, 0))
        starts = np.empty((n.value, 3), np.int32)
        check(self._lib.cfb_patch_grid(self._h, cz, cy, cx, C.byref(n), _ptr(starts), n.value))
        return starts

    def output_shape(self, chunk_zyx) -> tuple:
        out = (C.c_int64 * 4)()
        check(self._lib.cfb_output_shape(self._h, *(int(v) for v in chunk_zyx), C.byref(out)))
        return tuple(out)

    @staticmethod
    def _dtype_code(dtype) -> int:
        if np.dtype(dtype) == np.uint8:
            return DTYPE_U8
        if np.dtype(dtype) == np.float32:
            return DTYPE_F32
        raise TypeError(f"input chunk dtype {dtype} is not supported on the device (uint8 or float32)")

    def infer_chunk_host(self, chunk: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        chunk = np.ascontiguousarray(chunk)
        if chunk.ndim != 3:
            raise ValueError("expected a (z, y, x) chunk")
        shape = self.output_shape(chunk.shape)
        if out is None:
            out = np.empty(shape, np.float32)
        assert out.shape == shape and out.dtype == np.float32 and out.flags.c_contiguous
        check(self._lib.cfb_infer_chunk_host(self._h, _ptr(chunk), self._dtype_code(chunk.dtype), *chunk.shape, _ptr(out)))
        return out

    def infer_chunk_device(self, d_in: int, dtype, chunk_zyx, d_out: int, stream: int = 0) -> None:
        check(self._lib.cfb_infer_chunk_device(self._h, C.c_void_p(d_in), self._dtype_code(dtype),
                                               *(int(v) for v in chunk_zyx), C.c_void_p(d_out), C.c_void_p(stream)))

    def infer_slab_device(self, d_in: int, dtype, chunk_zyx, zrow_begin: int, zrow_end: int, d_out: int, d_weight: int,
                          stream: int = 0) -> None:
        check(self._lib.cfb_infer_slab_device(self._h, C.c_void_p(d_in), self._dtype_code(dtype),
                                              *(int(v) for v in chunk_zyx), int(zrow_begin), int(zrow_end),
                                              C.c_void_p(d_out), C.c_void_p(d_weight), C.c_void_p(stream)))

    def normalize_device(self, d_out: int, d_weight: int, czyx, stream: int = 0, weight_is_inverse: bool = False,
                         all_zero_input: bool = False) -> None:
        check(self._lib.cfb_normalize_device(self._h, C.c_void_p(d_out), C.c_void_p(d_weight), int(bool(weight_is_inverse)),
                                             *(int(v) for v in czyx), int(bool(all_zero_input)), C.c_void_p(stream)))

    def slab_nonzero(self, stream: int = 0) -> bool:
        flag = C.c_int32()
        check(self._lib.cfb_slab_nonzero(self._h, C.byref(flag), C.c_void_p(stream)))
        return bool(flag.value)

    def weight_volume_device(self, chunk_zyx, z_begin: int, z_end: int, d_weight: int, invert: bool = False, stream: int = 0) -> None:
        check(self._lib.cfb_weight_volume_device(self._h, *(int(v) for v in chunk_zyx), int(z_begin), int(z_end), int(bool(invert)),
                                                 C.c_void_p(d_weight), C.c_void_p(stream)))

    def patch_forward_host(self, patches: np.ndarray) -> np.ndarray:
        patches = np.ascontiguousarray(patches, dtype=np.float32)
        if patches.ndim != 5 or patches.shape[1:] != (1,) + self.input_patch_size:
            raise ValueError(f"expected input patches of shape (batch, 1, {self.input_patch_size}), got {patches.shape}")
        b = patches.shape[0]
        out = np.empty((b, self.num_output_channels) + self.output_patch_size, np.float32)
        check(self._lib.cfb_patch_forward_host(self._h, _ptr(patches), b, _ptr(out)))
        return out

    # plugin level (user-supplied patch backends)
    def plugin_begin(self, chunk: np.ndarray) -> None:
        chunk = np.ascontiguousarray(chunk)
        check(self._lib.cfb_plugin_begin(self._h, _ptr(chunk), self._dtype_code(chunk.dtype), *chunk.shape))

    def plugin_extract(self, first: int, nb: int, out: np.ndarray) -> None:
        assert out.dtype == np.float32 and out.flags.c_contiguous
        if out.shape != (nb, 1) + self.input_patch_size:
            raise ValueError(f"patch buffer must have shape {(nb, 1) + self.input_patch_size}, got {out.shape}")
        check(self._lib.cfb_plugin_extract(self._h, int(first), int(nb), _ptr(out)))

    def plugin_blend(self, first: int, nb: int, masked: np.ndarray) -> None:
        """`masked`: what the user's patch backend returned for patches [first, first+nb) -- already cropped to the output
        patch and bump-masked.  The native side reads nb*C*prod(output_patch_size) floats, so the shape is checked here
        (the reference fails with a numpy broadcasting error on a wrong shape)."""
        masked = np.asarray(masked)
        want = (nb, self.num_output_channels) + self.output_patch_size
        if masked.shape != want:
            raise ValueError(f"the patch backend must return an array of shape {want} (batch, channels, cropped output patch); "
                             f"got {masked.shape}")
        masked = np.ascontiguousarray(masked, dtype=np.float32)
        check(self._lib.cfb_plugin_blend(self._h, int(first), int(nb), _ptr(masked)))

    def plugin_end(self, out: np.ndarray) -> None:
        check(self._lib.cfb_plugin_end(self._h, _ptr(out)))

    def last_timing(self) -> dict:
        ms = (C.c_float * 5)()
        n = C.c_int64()
        check(self._lib.cfb_last_timing(self._h, C.byref(ms), C.byref(n)))
        return dict(total_ms=ms[0], convnet_ms=ms[1], blend_normalize_ms=ms[2], h2d_ms=ms[3], d2h_ms=ms[4],
                    launches=n.value)

    def set_profiling(self, enabled: bool) -> None:
        check(self._lib.cfb_set_profiling(self._h, int(bool(enabled))))

    def layer_timing(self) -> dict:
        """kernel class -> (total ms, launches) since profiling was enabled."""
        cap = 64
        names = (C.c_char * 32 * cap)()
        ms = (C.c_float * cap)()
        launches = (C.c_int64 * cap)()
        n = C.c_int32()
        check(self._lib.cfb_layer_timing(self._h, cap, C.byref(n), C.cast(names, C.c_void_p), C.cast(ms, C.c_void_p),
                                         C.cast(launches, C.c_void_p)))
        return {names[i].value.decode(): (float(ms[i]), int(launches[i])) for i in range(n.value)}

    def debug_net_forward(self, patch: np.ndarray, cnet: int) -> np.ndarray:
        patch = np.ascontiguousarray(patch, dtype=np.float32)
        out = np.empty((cnet,) + self.input_patch_size, np.float32)
        check(self._lib.cfb_debug_net_forward_host(self._h, _ptr(patch), _ptr(out)))
        return out

    def debug_conv3(self, x: np.ndarray, w: np.ndarray, b: np.ndarray, relu: bool) -> np.ndarray:
        x = np.ascontiguousarray(x, np.float32); w = np.ascontiguousarray(w, np.float32); b = np.ascontiguousarray(b, np.float32)
        cin, z, y, xx = x.shape
        cout = w.shape[0]
        out = np.empty((cout, z, y, xx), np.float32)
        check(self._lib.cfb_debug_conv3_host(self._h, _ptr(x), cin, z, y, xx, _ptr(w), _ptr(b), cout, int(relu), _ptr(out)))
        return out
