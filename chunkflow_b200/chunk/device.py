"""A chunk that lives in GPU memory between operators (SURVEY.md section 8 f3).

``DeviceChunk`` wraps a CUDA ``torch.Tensor`` (the memory container only) with the ``voxel_offset`` / ``voxel_size``
bookkeeping of the reference's ``Chunk`` and mirrors, name for name, the reference methods that sit either side of the
``inference`` operator in a pipeline -- each one a hand-written kernel behind the C ABI (``include/chunkflow_b200.h``,
``csrc/operators.cu``), bit-identical to the reference's numpy code:

    normalize_contrast   reference chunk/image/base.py:93-132          (Image)
    maskout              reference chunk/base.py:811-829                (Chunk; ``mask.maskout(chunk)`` modifies ``chunk``)
    crop_margin          reference chunk/base.py:691-726                (Chunk)
    quantize             reference chunk/affinity_map/base.py:33-57     (AffinityMap)
    connected_component  reference chunk/base.py:128-137                (Chunk -> cc3d)
    agglomerate          reference plugins/agglomerate.py:8-48          (plugin -> waterz)
    evaluate             reference chunk/segmentation.py:33-67          (Segmentation -> gala)

so that ``create-chunk | normalize-contrast | inference | crop-margin | quantize`` moves the image to the GPU once and
brings a uint8 thumbnail (or nothing) back instead of the 12-byte-per-voxel affinity map.  There is no CPU fallback.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from .. import _native
from ..lib.cartesian_coordinate import Cartesian, to_cartesian
from .base import Chunk


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("chunkflow_b200.DeviceChunk needs a CUDA device (there is no CPU fallback)")
    return torch


def _dtype_code(t) -> int:
    torch = _torch()
    if t.dtype in (torch.uint8, torch.bool):
        return _native.DTYPE_U8
    if t.dtype == torch.float32:
        return _native.DTYPE_F32
    raise TypeError(f"DeviceChunk operators support uint8/bool and float32, got {t.dtype}")


def mask_array_for(chunk_dtype, mask: np.ndarray) -> np.ndarray:
    """Host-side conversion of a mask of any dtype numpy accepts in ``chunk *= mask`` (reference chunk/base.py:811-829)
    to one of the two mask dtypes the kernel takes, WITHOUT changing the result:

    * uint8 chunk: numpy multiplies in the wider unsigned type and casts back modulo 256, which equals multiplying by
      ``mask mod 256`` -> uint8 mask (signed / float masks are refused by numpy's 'same_kind' rule, and here);
    * float32 chunk: an integer mask is converted by numpy to float64, the product rounded to float32; for |mask| < 2**24
      that is the float32 product with the exactly converted mask -> float32 mask.  float64 masks are refused (the
      double-precision product does not round like a float32 one)."""
    chunk_dtype = np.dtype(chunk_dtype)
    mask = np.asarray(mask)
    if mask.dtype in (np.dtype(np.uint8), np.dtype(bool)) or (mask.dtype == np.float32 and chunk_dtype == np.float32):
        return np.ascontiguousarray(mask)
    if chunk_dtype == np.uint8:
        if mask.dtype.kind != "u":
            raise TypeError(f"numpy cannot cast {mask.dtype} to uint8 in place (same_kind); neither do we")
        return np.ascontiguousarray(mask.astype(np.uint8))  # wraps modulo 256
    if chunk_dtype == np.float32:
        if mask.dtype.kind not in "ui":
            raise TypeError(f"a {mask.dtype} mask on a float32 chunk is not supported (product rounds differently)")
        if mask.size and int(np.abs(mask.astype(np.int64)).max()) >= 2 ** 24:
            raise TypeError("integer mask values must be below 2**24 to be exact in float32")
        return np.ascontiguousarray(mask.astype(np.float32))
    raise TypeError(f"unsupported chunk dtype {chunk_dtype}")


EVALUATE_INITIAL_SLOTS = 1 << 20   # contingency-table slots of the first attempt; grown eightfold while the pairs overflow it


class DeviceChunk:
    def __init__(self, tensor, voxel_offset=None, voxel_size=None, layer_type: Optional[str] = None):
        torch = _torch()
        assert isinstance(tensor, torch.Tensor) and tensor.is_cuda, "DeviceChunk wraps a CUDA tensor"
        assert tensor.ndim in (3, 4)
        self.tensor = tensor.contiguous()
        self.voxel_offset = to_cartesian(voxel_offset) if voxel_offset is not None else Cartesian(0, 0, 0)
        self.voxel_size = to_cartesian(voxel_size) if voxel_size is not None else None
        self.layer_type = layer_type

    # ---- host <-> device -------------------------------------------------------------------
    @classmethod
    def from_chunk(cls, chunk: Chunk, device="cuda:0") -> "DeviceChunk":
        torch = _torch()
        arr = np.ascontiguousarray(chunk.array)
        return cls(torch.from_numpy(arr).to(device), voxel_offset=chunk.voxel_offset, voxel_size=chunk.voxel_size,
                   layer_type=getattr(chunk, "_layer_type", None))

    @classmethod
    def mask_from_chunk(cls, mask: Chunk, like: "DeviceChunk") -> "DeviceChunk":
        """A mask chunk of any numpy dtype (the reference's own test uses uint32) for ``maskout`` of ``like``:
        converted on the host by :func:`mask_array_for`, then uploaded to ``like``'s GPU."""
        torch = _torch()
        target = np.uint8 if like.tensor.dtype == torch.uint8 else np.float32
        arr = mask_array_for(target, mask.array)
        return cls(torch.from_numpy(arr).to(like.tensor.device), voxel_offset=mask.voxel_offset, voxel_size=mask.voxel_size)

    @classmethod
    def from_labels(cls, labels: np.ndarray, device="cuda:0", voxel_offset=None, voxel_size=None) -> "DeviceChunk":
        """A (z,y,x) uint32 / uint64 label volume, uploaded as int32 / int64 with the same bits (torch's unsigned types
        have few operations)."""
        torch = _torch()
        signed = {np.dtype(np.uint32): np.int32, np.dtype(np.uint64): np.int64}[np.dtype(labels.dtype)]
        t = torch.from_numpy(np.ascontiguousarray(labels).view(signed)).to(device)
        return cls(t, voxel_offset=voxel_offset, voxel_size=voxel_size, layer_type="segmentation")

    def to_chunk(self) -> Chunk:
        return Chunk(self.tensor.cpu().numpy(), voxel_offset=self.voxel_offset, voxel_size=self.voxel_size)

    @property
    def shape(self):
        return tuple(self.tensor.shape)

    @property
    def dtype(self):
        return self.tensor.dtype

    def _czyx(self):
        s = self.shape
        return (1,) + s if len(s) == 3 else s

    def _stream(self) -> int:
        return _torch().cuda.current_stream(self.tensor.device).cuda_stream

    def _on_device(self):
        return _torch().cuda.device(self.tensor.device)

    # ---- Image.normalize_contrast ---------------------------------------------------------
    def normalize_contrast(self, lower_clip_fraction: float = 0.01, upper_clip_fraction: float = 0.01, minval: int = 1,
                           maxval: int = 255, per_section: bool = True) -> None:
        """In place, like the reference (including its quirks: the whole-array pass also runs after the per-section pass,
        and ``per_section=False`` does nothing)."""
        torch = _torch()
        assert self.tensor.dtype == torch.uint8 and self.tensor.ndim == 3, "normalize_contrast works on a (z,y,x) uint8 image"
        with self._on_device():
            _native.normalize_contrast_device(self.tensor.data_ptr(), self.shape, lower_clip_fraction, upper_clip_fraction,
                                              minval, maxval, per_section, self._stream())

    # ---- Chunk.maskout: self is the MASK, ``chunk`` is modified in place ---------------------
    def maskout(self, chunk: "DeviceChunk") -> None:
        assert chunk.voxel_size is not None and self.voxel_size is not None  # reference chunk/base.py:814-815
        assert all(m >= c for m, c in zip(self.voxel_size, chunk.voxel_size))
        assert all(m % c == 0 for m, c in zip(self.voxel_size, chunk.voxel_size)), "the voxel size should be divisible"
        factor = tuple(m // c for m, c in zip(self.voxel_size, chunk.voxel_size))
        assert self.tensor.ndim == 3
        assert tuple(chunk.shape[-3:]) == tuple(s * f for s, f in zip(self.shape, factor)), \
            "chunk size must equal mask size times the voxel-size factor"
        with self._on_device():
            _native.maskout_device(chunk.tensor.data_ptr(), _dtype_code(chunk.tensor), chunk._czyx(), self.tensor.data_ptr(),
                                   _dtype_code(self.tensor), factor, chunk._stream())

    # ---- Chunk.crop_margin ----------------------------------------------------------------
    def crop_margin(self, margin_size: Sequence[int]) -> "DeviceChunk":
        torch = _torch()
        m = tuple(int(v) for v in margin_size)
        if len(m) == 3:
            m6 = m + m
        elif len(m) == 6:
            m6 = m
        else:
            raise ValueError('only support 3 or 6 elements.')  # reference chunk/base.py:719
        c, z, y, x = self._czyx()
        out_sp = (z - m6[0] - m6[3], y - m6[1] - m6[4], x - m6[2] - m6[5])
        out_shape = out_sp if self.tensor.ndim == 3 else (c,) + out_sp
        dst = torch.empty(out_shape, dtype=self.tensor.dtype, device=self.tensor.device)
        with self._on_device():
            _native.crop_margin_device(self.tensor.data_ptr(), _dtype_code(self.tensor), (c, z, y, x), m6, dst.data_ptr(),
                                       self._stream())
        offset = tuple(o + mm for o, mm in zip(self.voxel_offset, m))  # the three lower margins (reference :721-722)
        return DeviceChunk(dst, voxel_offset=offset, voxel_size=self.voxel_size)

    # ---- AffinityMap.quantize -------------------------------------------------------------
    def quantize(self, mode: str = 'xy') -> "DeviceChunk":
        torch = _torch()
        assert self.tensor.dtype == torch.float32 and self.tensor.ndim == 4, "quantize works on a (c,z,y,x) float32 affinity map"
        if mode == 'xy':
            code = _native.QUANTIZE_XY
        elif mode == 'z':
            code = _native.QUANTIZE_Z
        else:
            raise ValueError(f'only support xy and z mode, but got {mode}')
        out = torch.empty(self.shape[1:], dtype=torch.uint8, device=self.tensor.device)
        with self._on_device():
            _native.quantize_device(self.tensor.data_ptr(), self.shape, code, out.data_ptr(), self._stream())
        return DeviceChunk(out, voxel_offset=self.voxel_offset, voxel_size=self.voxel_size)

    # ---- Chunk.connected_component ---------------------------------------------------------
    def connected_component(self, threshold: float = None, connectivity: int = 6) -> "DeviceChunk":
        """Threshold the map and label its connected components (reference chunk/base.py:128-137: ``Chunk.threshold`` --
        ``array > threshold`` -- for non-segmentation chunks, then ``cc3d.connected_components(seg, connectivity)``).
        (z,y,x) or (1,z,y,x) float32 map with a threshold, or a uint8 / int32 / uint32 segmentation; returns a (z,y,x) uint32
        segmentation whose components are numbered 1..N in raster order of their first voxel, like cc3d."""
        torch = _torch()
        t = self.tensor
        if t.ndim == 4:
            assert t.shape[0] == 1   # reference base.py:730-732
            t = t[0]
        is_seg = t.dtype in (torch.uint8, torch.bool, torch.int32, torch.uint32) or self.layer_type == "segmentation"
        thr = 0.0
        if not is_seg and threshold is not None:
            assert t.dtype == torch.float32, "thresholding works on a float32 map"
            code, thr = _native.DTYPE_F32, float(threshold)
        elif t.dtype in (torch.uint8, torch.bool):
            code = _native.DTYPE_U8
        elif t.dtype in (torch.int32, torch.uint32):
            code = _native.DTYPE_U32
        else:
            raise TypeError(f"connected_component: {t.dtype} without a threshold is not a segmentation (uint8 / int32 / uint32)")
        if connectivity not in (6, 18, 26):
            raise ValueError("connectivity must be 6, 18 or 26")
        t = t.contiguous()
        labels = torch.empty(t.shape, dtype=torch.int32, device=t.device)   # uint32 values (torch has no full uint32 support)
        work = torch.empty(_native.connected_components_workspace(t.shape), dtype=torch.uint8, device=t.device)
        with self._on_device():
            self.num_components = _native.connected_components_device(t.data_ptr(), code, tuple(t.shape), thr, connectivity,
                                                                      labels.data_ptr(), work.data_ptr(), self._stream())
        del work
        out = DeviceChunk(labels.view(torch.uint32) if hasattr(torch, "uint32") else labels, voxel_offset=self.voxel_offset,
                          voxel_size=self.voxel_size, layer_type="segmentation")
        out.num_components = self.num_components
        return out

    # ---- plugins/agglomerate.py: watershed fragments + mean-affinity agglomeration --------------
    def _affinity_tensor(self):
        torch = _torch()
        t = self.tensor
        assert t.ndim == 4 and t.shape[0] == 3 and t.dtype == torch.float32, \
            "an affinity map is a (3, z, y, x) float32 chunk (the reference converts with np.ascontiguousarray(affs, dtype=float32))"
        if t.numel() // 3 >= 2 ** 32 - 1:
            raise ValueError("more than 2^32 - 1 voxels")
        return t

    def watershed(self, aff_threshold_low: float = 0.001, aff_threshold_high: float = 0.9999,
                  flip_channel: bool = True) -> "DeviceChunk":
        """Fragments of the affinity map by steepest-ascent watershed (what ``waterz.agglomerate`` computes first when no
        fragments are passed, reference plugins/agglomerate.py:36-41): (z,y,x) uint32, basins numbered 1..N in raster order
        of their first voxel, 0 where no affinity exceeds ``aff_threshold_low``.  ``flip_channel``: the channels are stored
        in chunkflow's order x, y, z (agglomerate.py:26-29); they are read in reverse, not copied."""
        torch = _torch()
        t = self._affinity_tensor()
        zyx = tuple(t.shape[1:])
        frag = torch.empty(zyx, dtype=torch.int32, device=t.device)   # uint32 values
        work = torch.empty(_native.watershed_workspace(zyx), dtype=torch.uint8, device=t.device)
        with self._on_device():
            n = _native.watershed_device(t.data_ptr(), flip_channel, zyx, aff_threshold_low, aff_threshold_high, frag.data_ptr(),
                                         work.data_ptr(), self._stream())
        del work
        out = DeviceChunk(frag.view(torch.uint32) if hasattr(torch, "uint32") else frag, voxel_offset=self.voxel_offset,
                          voxel_size=self.voxel_size, layer_type="segmentation")
        out.num_components = n
        return out

    def region_graph(self, fragments: "DeviceChunk", flip_channel: bool = True, num_fragments: Optional[int] = None):
        """(u, v, sum_fixed, count) host arrays, one entry per pair of touching fragments, sorted by (u, v): the sum (2^-30
        fixed point) and number of the affinities on the faces between them (waterz's region graph with MeanAffinity
        statistics).  The hash table is sized from the fragment count and grown on overflow."""
        torch = _torch()
        t = self._affinity_tensor()
        f = fragments.tensor
        assert tuple(f.shape) == tuple(t.shape[1:]) and f.dtype in (torch.int32, torch.uint32) and f.device == t.device
        if num_fragments is None:
            num_fragments = getattr(fragments, "num_components", None)
        if num_fragments is None:
            num_fragments = int(f.view(torch.int32).max().item()) if f.numel() else 0
        slots = 1 << 16
        while slots < 16 * num_fragments:
            slots <<= 1
        with self._on_device():
            while True:
                work = torch.empty(_native.region_graph_workspace(slots), dtype=torch.uint8, device=t.device)
                try:
                    n = _native.region_graph_device(t.data_ptr(), flip_channel, f.data_ptr(), tuple(f.shape), work.data_ptr(), slots,
                                                    self._stream())
                    if 2 * n <= slots:
                        break
                except _native.NativeError as err:
                    if err.code != _native.ERR_CAPACITY:
                        raise
                del work
                slots <<= 2          # too full (or more than half full: long probe sequences): a larger table
                if slots >= 1 << 31:
                    raise RuntimeError("region graph: more fragment pairs than the table can hold")
            return _native.region_graph_read(work.data_ptr(), slots, n, self._stream())

    def agglomerate(self, threshold: float = 0.7, aff_threshold_low: float = 0.001, aff_threshold_high: float = 0.9999,
                    fragments: Optional["DeviceChunk"] = None, flip_channel: bool = True) -> "DeviceChunk":
        """Mean-affinity agglomeration including the watershed step (reference plugins/agglomerate.py:8-48 ->
        ``waterz.agglomerate`` with ``OneMinus<MeanAffinity<RegionGraphType, ScoreValue>>``): fragments (watershed, unless
        given) -> region graph -> merge edges in order of increasing ``1 - mean affinity`` until ``threshold`` -> relabel.
        The voxel passes are CUDA kernels; the merge loop over the fragment graph runs in the native library on the host
        (as waterz's does).  Returns a (z,y,x) uint32 segmentation whose ids are the surviving fragment ids."""
        torch = _torch()
        t = self._affinity_tensor()
        if fragments is None:
            fragments = self.watershed(aff_threshold_low, aff_threshold_high, flip_channel)
        f = fragments.tensor
        if f.dtype not in (torch.int32, torch.uint32):
            raise TypeError("fragments must be an int32 / uint32 segmentation on the device")
        num = getattr(fragments, "num_components", None)
        if num is None:
            num = int(f.view(torch.int32).max().item()) if f.numel() else 0
        if num < 0:
            raise ValueError("fragment ids must be below 2^31")
        u, v, s, c = self.region_graph(fragments, flip_channel, num)
        root = _native.agglomerate_edges_host(num + 1, u, v, s, c, threshold)
        d_root = torch.from_numpy(root.view(np.int32)).to(t.device)
        seg = torch.empty(f.shape, dtype=torch.int32, device=t.device)
        with self._on_device():
            _native.relabel_device(f.data_ptr(), f.numel(), d_root.data_ptr(), root.size, seg.data_ptr(), self._stream())
            _torch().cuda.current_stream(t.device).synchronize()   # d_root is released below
        out = DeviceChunk(seg.view(torch.uint32) if hasattr(torch, "uint32") else seg, voxel_offset=self.voxel_offset,
                          voxel_size=self.voxel_size, layer_type="segmentation")
        out.num_fragments, out.num_edges = num, int(u.size)
        out.num_components = int(np.count_nonzero(root[1:] == np.arange(1, root.size, dtype=np.uint32)))
        return out

    # ---- Segmentation.evaluate (reference chunk/segmentation.py:33-67 -> lib/gala/evaluate.py) ------------------------
    def _label_tensor(self, what: str):
        """The labels as a contiguous 4- or 8-byte tensor and its native dtype code; ids are read as unsigned, narrower
        integer types are widened (bijections that keep 0 change no score)."""
        torch = _torch()
        t = self.tensor
        if t.ndim == 4:
            if t.shape[0] != 1:
                raise ValueError(f"{what}: a segmentation has one channel, not {t.shape[0]}")
            t = t[0]
        if t.is_floating_point() or t.is_complex():
            raise TypeError(f"{what} must be an integer label volume, not {t.dtype}")
        if t.element_size() < 4:
            t = t.to(torch.int32)
        t = t.contiguous()
        if t.data_ptr() % 16:
            t = t.clone()
        return t, (_native.DTYPE_U64 if t.element_size() == 8 else _native.DTYPE_U32)

    def _contingency(self, groundtruth: "DeviceChunk"):
        """Builds the contingency table of (self, groundtruth) on the device -> (workspace, slots, entries, voxels)."""
        torch = _torch()
        s, s_code = self._label_tensor("the segmentation")
        g, g_code = groundtruth._label_tensor("the ground truth")
        if tuple(s.shape) != tuple(g.shape):
            raise ValueError(f"the ground truth has shape {tuple(g.shape)}, the segmentation {tuple(s.shape)}")
        if s.device != g.device:
            raise ValueError("the segmentation and the ground truth must be on the same GPU")
        n = s.numel()
        slots = EVALUATE_INITIAL_SLOTS
        most = 4
        while most < 2 * n:   # a table never holds more pairs than voxels
            most <<= 1
        slots = max(2, min(slots, most))
        with self._on_device():
            while True:
                work = torch.empty(_native.contingency_workspace(slots), dtype=torch.uint8, device=s.device)
                try:
                    entries = _native.contingency_device(s.data_ptr(), s_code, g.data_ptr(), g_code, n, work.data_ptr(), slots,
                                                         work.numel(), self._stream())
                    return work, slots, entries, n
                except _native.NativeError as err:
                    if err.code != _native.ERR_CAPACITY or slots >= most:
                        raise
                del work
                slots = min(slots << 3, most)   # more pairs than half the slots: a larger table

    def evaluate(self, groundtruth: "DeviceChunk", size_threshold: float = 1000) -> dict:
        """The reference's ``Segmentation.evaluate`` dict (``rand_index``, ``adjusted_rand_index``,
        ``variation_of_information``, ``fowlkes_mallows_index``, ``edit_distance``) of this segmentation against
        ``groundtruth``, both (z,y,x) integer volumes on the same GPU.  One pass over both volumes builds the contingency
        table; a reduction on the device turns it into exact integer sums; the scores are finished on the host."""
        from .segmentation import scores_from_sums
        work, slots, entries, n = self._contingency(groundtruth)
        with self._on_device():
            sums = _native.contingency_scores(work.data_ptr(), slots, n, entries, float(size_threshold), work.numel(), self._stream())
        return scores_from_sums(sums)

    def contingency_table(self, groundtruth: "DeviceChunk"):
        """(seg_ids, gt_ids, counts) uint64 host arrays: the number of voxels of every label pair that occurs, sorted by
        (seg id, gt id); signed ids appear as their unsigned bit patterns."""
        work, slots, entries, _ = self._contingency(groundtruth)
        with self._on_device():
            return _native.contingency_read(work.data_ptr(), slots, entries, work.numel(), self._stream())

    def __repr__(self):
        return f"DeviceChunk(shape={self.shape}, dtype={self.dtype}, voxel_offset={tuple(self.voxel_offset)}, device={self.tensor.device})"
