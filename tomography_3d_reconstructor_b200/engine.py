"""Device-side engine: thin Python over the C ABI (include/t3d.h).

PyTorch is used only for device buffers, streams and host<->device copies; every arithmetic step is a
kernel of libt3d.so.  Nothing in this module computes on the CPU and nothing falls back to it.
"""
from __future__ import annotations

import ctypes
import weakref
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import T3DError, check


class T3DUnavailable(T3DError):
    """libt3d.so or a CUDA device is missing.  Never swallowed by the reference-style `except Exception`."""


def _require_cuda() -> torch.device:
    if not torch.cuda.is_available():
        raise T3DUnavailable("a CUDA device is required: this package has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _L():
    try:
        return _lib.load()
    except T3DError as e:  # missing shared object
        raise T3DUnavailable(str(e)) from None


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]) -> Optional[ctypes.c_void_p]:
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def words_per_row(W: int) -> int:
    """Row stride in 32-bit words: ceil(W/32) rounded up to a multiple of 4 (16-byte aligned rows)."""
    return (((W + 31) // 32) + 3) & ~3


# scipy.ndimage._filters._gaussian_kernel1d(sigma=0.5, order=0, radius=2), restated with numpy so the three
# weights are bit-identical to what gaussian_filter(sigma=0.5) uses (surface_extractor.py:50-51)
def gaussian_weights_sigma_half() -> np.ndarray:
    sigma, radius = 0.5, int(4.0 * 0.5 + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    phi = phi / phi.sum()
    return np.array([phi[2], phi[1], phi[0]], dtype=np.float64)  # centre, +-1, +-2


_W3 = gaussian_weights_sigma_half()
_W3_C = (ctypes.c_double * 3)(*_W3.tolist())


# ----------------------------------------------------------------------------------------------------------
# device containers
# ----------------------------------------------------------------------------------------------------------
class DeviceVolume:
    """Bit-packed occupancy (Z, H, wpr) int32 on the device + lazily cached reductions."""

    __slots__ = ("bits", "Z", "H", "W", "_counts", "_bbox", "memo", "__weakref__")

    def __init__(self, bits: torch.Tensor, Z: int, H: int, W: int, counts: Optional[torch.Tensor] = None):
        self.bits, self.Z, self.H, self.W = bits, Z, H, W
        self._counts = counts  # device int64 (Z,) or host np.int64 once fetched
        self._bbox = None
        self.memo = {}         # results derived from this (immutable) volume: smoothing, extraction (SURVEY.md 8f-2)

    @property
    def shape(self) -> Tuple[int, int, int]:
        return (self.Z, self.H, self.W)

    # per-slice np.sum(voxel_data[z]) (volume_calculator.py:31-33), exact integers
    def slice_counts(self) -> np.ndarray:
        if isinstance(self._counts, np.ndarray):
            return self._counts
        if self._counts is None:
            self._run_stats()
        c = self._counts.cpu().numpy().astype(np.int64)
        self._counts = c
        return c

    def _run_stats(self) -> None:
        dev = self.bits.device
        counts = torch.empty(self.Z, dtype=torch.int64, device=dev) if self._counts is None else None
        bbox = torch.empty(6, dtype=torch.int32, device=dev)
        check(_L().t3d_volume_stats(_p(self.bits), self.Z, self.H, self.W, _p(counts), _p(bbox), _stream()),
              "t3d_volume_stats")
        if self._counts is None:
            self._counts = counts
        self._bbox = bbox

    # device-side handles (no synchronisation): used by pipeline.reconstruct to fetch everything in one copy
    def counts_tensor(self) -> torch.Tensor:
        if self._counts is None:
            self._run_stats()
        if isinstance(self._counts, np.ndarray):
            return torch.from_numpy(self._counts).to(self.bits.device)
        return self._counts

    def bbox_tensor(self) -> torch.Tensor:
        if self._bbox is None:
            self._run_stats()
        if isinstance(self._bbox, torch.Tensor):
            return self._bbox
        b = self._bbox if self._bbox else (0x7fffffff, -1) * 3
        return torch.tensor(b, dtype=torch.int32, device=self.bits.device)

    def set_host_stats(self, counts: np.ndarray, bbox) -> None:
        self._counts = np.asarray(counts, dtype=np.int64)
        if bbox is not None:
            b = tuple(int(v) for v in bbox)
            self._bbox = b if b[1] >= 0 else ()

    def bbox(self) -> Optional[Tuple[int, int, int, int, int, int]]:
        """(zmin, zmax, ymin, ymax, xmin, xmax) of the set voxels, None if the volume is empty."""
        if self._bbox is None:
            self._run_stats()
        if isinstance(self._bbox, torch.Tensor):
            b = tuple(int(v) for v in self._bbox.cpu().tolist())
            self._bbox = b if b[1] >= 0 else ()
        return self._bbox if self._bbox else None

    def to_host(self) -> np.ndarray:
        """numpy bool (Z, H, W): unpack on the device, copy through pinned memory."""
        out = torch.empty((self.Z, self.H, self.W), dtype=torch.uint8, device=self.bits.device)
        check(_L().t3d_unpack_bits(_p(self.bits), self.Z, self.H, self.W, _p(out), _stream()), "t3d_unpack_bits")
        host = torch.empty((self.Z, self.H, self.W), dtype=torch.bool, pin_memory=True)
        host.view(torch.uint8).copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host.numpy()


def download(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> numpy array backed by pinned host memory (DMA at PCIe speed; torch's caching host allocator
    recycles the pinned blocks).  A plain `.cpu()` goes through pageable memory at a fraction of the bandwidth."""
    t = t.contiguous()
    host = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    host.copy_(t, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return host.numpy()


class DeviceMesh:
    """Mesh on the device.  After an asynchronous canonicalisation the arrays are capacity-sized and the true sizes
    live in `counts_dev` until resolve() (one D2H copy) or set_sizes() trims them."""

    __slots__ = ("_verts", "_faces", "counts_dev", "n_ambiguous", "n_exact", "_measures", "raw", "n_active", "n_raw", "n_z",
                 "normal_src", "canon_map", "_normals", "__weakref__")

    def __init__(self, verts: torch.Tensor, faces: torch.Tensor, n_ambiguous: int = 0, n_exact: int = 0,
                 counts_dev: Optional[torch.Tensor] = None):
        self._verts, self._faces = verts, faces
        self.counts_dev = counts_dev
        self.n_ambiguous, self.n_exact = n_ambiguous, n_exact
        self._measures = None
        self.raw = None  # (raw verts, raw faces) of an asynchronous canonicalisation, until the sizes are known
        self.n_active = 0        # active 32-voxel words / raw (vertices, faces): capacity hints for the fused path
        self.n_raw = (0, 0)
        # field-gradient normals (extract_surface(normals=True)): what the kernel reads -- field source, vertex keys, z map --
        # and the raw -> canonical map of the canonicalisation (canonical_map(); None: raw vertex order)
        self.normal_src = None
        self.canon_map = None
        self._normals = None

    def set_sizes(self, n_verts: int, n_faces: int, unverified: int = 0) -> None:
        """Trim the capacity-sized arrays.  unverified != 0: the fast ordering failed its device-side check, redo the
        canonicalisation with the general three-key sort (degenerate inputs only)."""
        if unverified and self.raw is not None:
            keep = {} if self.normal_src is not None else None
            self._verts, self._faces = canonicalize(self.raw[0], self.raw[1], self._faces.dtype == torch.int64, True, False, keep=keep)
            if keep is not None:
                self.canon_map = keep["map"]
        else:
            self._verts, self._faces = self._verts[:n_verts], self._faces[:n_faces]
        self.counts_dev = None
        self.raw = None

    def resolve(self) -> "DeviceMesh":
        if self.counts_dev is not None:
            v2, f2, bad = (int(c) for c in self.counts_dev.cpu().tolist())
            self.set_sizes(v2, f2, bad)
        return self

    @property
    def verts(self) -> torch.Tensor:
        return self.resolve()._verts

    @property
    def faces(self) -> torch.Tensor:
        return self.resolve()._faces

    @property
    def normals(self) -> Optional[torch.Tensor]:
        """Field-gradient unit normals, device float32 (V', 3) [z, y, x], row i for vertex i (DESIGN.md §2); None unless the
        mesh was extracted with normals=True."""
        if self._normals is None and self.normal_src is not None:
            self._normals = mesh_normals(self)
        return self._normals

    def measures(self) -> Tuple[float, float]:
        """(signed volume, area), float64 accumulation on the device."""
        if self._measures is None:
            self._measures = mesh_measure(self.verts, self.faces)
        return self._measures


# ----------------------------------------------------------------------------------------------------------
# identity registry: host ndarray handed to the caller -> device object it was materialised from
# ----------------------------------------------------------------------------------------------------------
class _Registry:
    def __init__(self):
        self._d = {}

    def register(self, arr: np.ndarray, obj) -> None:
        key = id(arr)

        def _drop(_ref, key=key, d=self._d):
            d.pop(key, None)

        self._d[key] = (weakref.ref(arr, _drop), obj)

    def lookup(self, arr):
        e = self._d.get(id(arr))
        if e is not None and e[0]() is arr:
            return e[1]
        return None


volumes = _Registry()
meshes = _Registry()

# Host arrays handed to the caller mirror a device object that later calls recognise by array identity (smooth -> extract
# -> volume never re-uploads).  That only holds while the array cannot change, so by default it is read-only; the
# reference returns ordinary writable arrays.  T3D_WRITABLE_OUTPUTS=1 (or engine.WRITABLE_OUTPUTS = True) hands out
# writable arrays instead and does not register them: every later call uploads what the array then contains.
import os as _os
WRITABLE_OUTPUTS = bool(_os.environ.get("T3D_WRITABLE_OUTPUTS"))


def publish(registry: "_Registry", arr: np.ndarray, obj) -> np.ndarray:
    if WRITABLE_OUTPUTS:
        try:
            arr.setflags(write=True)
        except ValueError:            # a view of memory numpy does not own (pinned staging buffer): hand out a copy
            arr = np.array(arr)
        return arr
    arr.setflags(write=False)
    registry.register(arr, obj)
    return arr


# ----------------------------------------------------------------------------------------------------------
# host -> device
# ----------------------------------------------------------------------------------------------------------
def _as_stack(mask_images) -> np.ndarray:
    """Return a (Z,H,W) 1-byte array without copying when the slices already lie back to back in memory."""
    if isinstance(mask_images, np.ndarray):
        arr = mask_images
        if arr.ndim != 3:
            raise ValueError("expected a (Z,H,W) stack")
    else:
        first = np.asarray(mask_images[0])
        n = len(mask_images)
        contiguous = first.ndim == 2 and first.flags.c_contiguous and first.dtype.itemsize == 1
        if contiguous:
            step = first.nbytes
            base = first.__array_interface__["data"][0]
            for k, m in enumerate(mask_images):
                if (not isinstance(m, np.ndarray) or m.shape != first.shape or m.dtype != first.dtype
                        or not m.flags.c_contiguous or m.__array_interface__["data"][0] != base + k * step):
                    contiguous = False
                    break
        if contiguous:
            buf = (ctypes.c_uint8 * (first.nbytes * n)).from_address(first.__array_interface__["data"][0])
            arr = np.frombuffer(buf, dtype=first.dtype).reshape((n,) + first.shape)
        else:
            arr = np.stack([np.asarray(m) for m in mask_images], axis=0)  # voxel_processor.py:46
    if arr.dtype == np.bool_:
        return arr.view(np.uint8)
    if arr.dtype == np.uint8:
        return arr
    return (arr != 0).view(np.uint8)


def upload_u8(stack_u8: np.ndarray) -> torch.Tensor:
    dev = _require_cuda()
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)  # read-only ndarray -> tensor (we only read it)
        t = torch.from_numpy(np.ascontiguousarray(stack_u8))
    return t.to(dev, non_blocking=True)


def pack(masks_u8_dev: torch.Tensor, threshold: int = 1) -> DeviceVolume:
    """image_loader.py:108 + np.stack (voxel_processor.py:46) on the device."""
    Z, H, W = (int(s) for s in masks_u8_dev.shape)
    bits = torch.empty((Z, H, words_per_row(W)), dtype=torch.int32, device=masks_u8_dev.device)
    check(_L().t3d_pack_masks(_p(masks_u8_dev), Z, H, W, int(threshold), _p(bits), _stream()), "t3d_pack_masks")
    return DeviceVolume(bits, Z, H, W)


_side_streams = {}


def side_stream(dev: torch.device) -> torch.cuda.Stream:
    """One auxiliary stream per device for work that is off the critical path (hole filling, bbox, measures)."""
    key = (dev.type, dev.index)
    st = _side_streams.get(key)
    if st is None:
        st = torch.cuda.Stream(device=dev)
        _side_streams[key] = st
    return st


def pack_and_close(masks_u8_dev: torch.Tensor, threshold: int = 1, close_ends: bool = True) -> DeviceVolume:
    """create_voxel_data on the device (voxel_processor.py:46-49).  The two end planes are packed first and their 2-D
    hole filling runs on a side stream while the bulk of the stack is being packed; the z gap fill joins both."""
    L = _L()
    Z, H, W = (int(s) for s in masks_u8_dev.shape)
    if not close_ends or Z < 3:
        dv = pack(masks_u8_dev, threshold)
        return close_volume_ends(dv) if close_ends else dv
    dev = masks_u8_dev.device
    wpr = words_per_row(W)
    bits = torch.empty((Z, H, wpr), dtype=torch.int32, device=dev)
    main = torch.cuda.current_stream()
    check(L.t3d_pack_masks(_p(masks_u8_dev[0]), 1, H, W, int(threshold), _p(bits[0]), _stream()), "t3d_pack_masks")
    check(L.t3d_pack_masks(_p(masks_u8_dev[Z - 1]), 1, H, W, int(threshold), _p(bits[Z - 1]), _stream()), "t3d_pack_masks")
    scratch = torch.empty(int(L.t3d_fill_holes_scratch_bytes(2, H, W)) // 4, dtype=torch.int32, device=dev)
    ends_packed = torch.cuda.Event()
    ends_packed.record(main)
    side = side_stream(dev)
    filled = torch.cuda.Event()
    with torch.cuda.stream(side):
        side.wait_event(ends_packed)
        check(L.t3d_fill_holes_2d(_p(bits), 2, (Z - 1) * H * wpr, H, W, _p(scratch), _stream()), "t3d_fill_holes_2d")
        filled.record(side)
    check(L.t3d_pack_masks(_p(masks_u8_dev[1]), Z - 2, H, W, int(threshold), _p(bits[1]), _stream()), "t3d_pack_masks")
    main.wait_event(filled)
    out = torch.empty_like(bits)
    counts = torch.empty(Z, dtype=torch.int64, device=dev)
    check(L.t3d_gap_fill(_p(bits), _p(out), None, None, Z, H, W, _p(counts), _stream()), "t3d_gap_fill")
    return DeviceVolume(out, Z, H, W, counts)


_copy_streams = {}
_capture_streams = {}
_stage_pool = None


def capture_stream(dev=None) -> "torch.cuda.Stream":
    """Stream for CUDA-graph capture ON THE GIVEN DEVICE.  torch.cuda.graph() otherwise captures on a class-level default
    stream created on whichever device used graphs first: on a second device of the same process the step would be
    captured (and its kernels launched) on the first device's stream."""
    idx = torch.cuda.current_device() if dev is None or getattr(dev, "index", None) is None else dev.index
    st = _capture_streams.get(idx)
    if st is None:
        st = _capture_streams[idx] = torch.cuda.Stream(device=idx)
    return st


def _pool():
    global _stage_pool
    if _stage_pool is None:
        from concurrent.futures import ThreadPoolExecutor
        _stage_pool = ThreadPoolExecutor(max_workers=min(8, (_os.cpu_count() or 2)))
    return _stage_pool


class PinnedRing:
    """Staging ring for mask lists as ImageLoader returns them (image_loader.py:97-109): Z separately allocated, pageable
    (H,W) bool / uint8 arrays.  A chunk of slices is copied into one of `slots` pinned buffers by a few host threads
    (numpy copies release the GIL) while the previous chunk's buffer is on its way to the device: the H2D copies run at
    PCIe speed from pinned memory and overlap the host-side gathering, and no (Z,H,W) host copy (np.stack) is made."""

    def __init__(self, H: int, W: int, chunk_planes: int, slots: int = 3):
        self.H, self.W, self.chunk = H, W, chunk_planes
        self.bufs = [torch.empty((chunk_planes, H, W), dtype=torch.uint8, pin_memory=True) for _ in range(slots)]
        self.views = [b.numpy() for b in self.bufs]
        self.events = [None] * slots
        self.k = 0

    def stage(self, source, a: int, b: int) -> torch.Tensor:
        """Slices [a, b) of `source` (list of arrays or a (Z,H,W) array) -> a pinned (b-a,H,W) uint8 tensor.  The caller
        records an event after its H2D copy with release()."""
        slot = self.k % len(self.bufs)
        self.k += 1
        if self.events[slot] is not None:
            self.events[slot].synchronize()        # the copy that last read this buffer has finished
        dst = self.views[slot]

        def one(z):
            m = np.asarray(source[z])
            if m.dtype == np.bool_:
                m = m.view(np.uint8)
            elif m.dtype != np.uint8:
                m = (m != 0).view(np.uint8)
            np.copyto(dst[z - a], m)

        n = b - a
        if n >= 4:
            list(_pool().map(one, range(a, b)))
        else:
            for z in range(a, b):
                one(z)
        self._slot = slot
        return self.bufs[slot][:n]

    def release(self, stream) -> None:
        ev = torch.cuda.Event()
        ev.record(stream)
        self.events[self._slot] = ev


_rings = {}


def _ring_for(H: int, W: int, chunk_planes: int) -> PinnedRing:
    key = (H, W, chunk_planes)
    r = _rings.get(key)
    if r is None:
        _rings.clear()                 # one shape at a time: pinned memory is a scarce resource
        r = _rings[key] = PinnedRing(H, W, chunk_planes)
    return r


def _is_pinned_stack(x) -> bool:
    if isinstance(x, torch.Tensor):
        return x.is_pinned()
    if isinstance(x, np.ndarray) and x.ndim == 3 and x.flags.c_contiguous and x.dtype.itemsize == 1:
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            return torch.from_numpy(x.view(np.uint8)).is_pinned()
    return False


def mask_source(mask_images):
    """(source, Z, H, W, pinned): `source[z]` is slice z; pinned = one contiguous pinned (Z,H,W) byte array (no staging)."""
    if isinstance(mask_images, (np.ndarray, torch.Tensor)):
        if mask_images.ndim != 3:
            raise ValueError("expected a (Z,H,W) stack")
        Z, H, W = (int(v) for v in mask_images.shape)
        return mask_images, Z, H, W, _is_pinned_stack(mask_images)
    # a list whose slices already lie back to back in memory is one array (e.g. views of a pinned stack): one pass over the
    # list (this runs per call on the host: ~1 us per slice)
    first = mask_images[0]
    if not isinstance(first, np.ndarray):
        first = np.asarray(first)
    if first.ndim != 2:
        raise ValueError("expected a list of (H,W) masks")
    n = len(mask_images)
    H, W = int(first.shape[0]), int(first.shape[1])
    if first.flags.c_contiguous and first.dtype.itemsize == 1 and first.dtype in (np.bool_, np.uint8):
        # in order and back to back iff every slice sits at its own offset from the first one
        step, addr, shape0, strides0, dt0 = first.nbytes, first.ctypes.data, first.shape, first.strides, first.dtype
        ok = True
        try:
            for k in range(1, n):
                m = mask_images[k]
                if m.ctypes.data != addr + k * step or m.strides != strides0 or m.shape != shape0 or m.dtype != dt0:
                    ok = False
                    break
        except AttributeError:        # not an ndarray
            ok = False
        if ok:
            buf = (ctypes.c_uint8 * (step * n)).from_address(addr)
            arr = np.frombuffer(buf, dtype=np.uint8).reshape((n, H, W))
            return arr, n, H, W, _is_pinned_stack(arr)
    return mask_images, n, H, W, False


def upload_masks(mask_images, out: Optional[torch.Tensor] = None, chunk_planes: int = 32) -> torch.Tensor:
    """Host masks (list or stack) -> uint8 (Z,H,W) on the device, enqueued on the current stream's timeline.  Pinned
    contiguous input: one async copy.  Anything else goes through the pinned staging ring in z-chunks."""
    dev = _require_cuda()
    src, Z, H, W, pinned = mask_source(mask_images)
    if out is None:
        out = torch.empty((Z, H, W), dtype=torch.uint8, device=dev)
    if pinned:
        t = src if isinstance(src, torch.Tensor) else torch.from_numpy(src.view(np.uint8))
        out.copy_(t.view(torch.uint8) if t.dtype != torch.uint8 else t, non_blocking=True)
        return out
    ring = _ring_for(H, W, chunk_planes)
    main = torch.cuda.current_stream()
    s_in, _ = _copy_stream_pair(dev)
    start = torch.cuda.Event()
    start.record(main)
    s_in.wait_event(start)
    for a in range(0, Z, chunk_planes):
        b = min(Z, a + chunk_planes)
        buf = ring.stage(src, a, b)
        with torch.cuda.stream(s_in):
            out[a:b].copy_(buf, non_blocking=True)
            ring.release(s_in)
    done = torch.cuda.Event()
    done.record(s_in)
    main.wait_event(done)
    return out


def _copy_stream_pair(dev: torch.device):
    key = (dev.type, dev.index)
    st = _copy_streams.get(key)
    if st is None:
        st = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
        _copy_streams[key] = st
    return st


def create_voxel_data_from_host(stack_u8, threshold: int = 1, close_ends: bool = True, chunk_planes: int = 32):
    """create_voxel_data (voxel_processor.py:36-54) for a host stack or list of masks, pipelined in z-chunks so that the upload of the
    masks (H2D), the kernels and the download of the resulting bool grid (D2H) overlap: PCIe is full duplex and the
    two directions use different copy engines.  Returns (DeviceVolume, numpy bool array in pinned memory).

    Chunk c is uploaded and packed while chunk c-1 is gap-filled (it needs one packed plane of chunk c), unpacked and
    downloaded.  Global slices 0 / Z-1 are hole-filled right after their chunk is packed, i.e. before any gap fill
    reads them, so the result is identical to the unpipelined path."""
    L = _L()
    dev = _require_cuda()
    source, Z, H, W, pinned = mask_source(stack_u8)
    wpr = words_per_row(W)
    if pinned:
        src = source if isinstance(source, torch.Tensor) else torch.from_numpy(source.view(np.uint8))
        ring = None
    else:           # pageable and / or scattered slices (what ImageLoader returns): pinned staging ring, no np.stack
        src, ring = None, _ring_for(H, W, chunk_planes)
    masks_dev = torch.empty((Z, H, W), dtype=torch.uint8, device=dev)
    bits = torch.empty((Z, H, wpr), dtype=torch.int32, device=dev)
    out_bits = torch.empty_like(bits)
    out_u8 = torch.empty((Z, H, W), dtype=torch.uint8, device=dev)
    counts = torch.empty(Z, dtype=torch.int64, device=dev)
    host = torch.empty((Z, H, W), dtype=torch.bool, pin_memory=True)
    host_u8 = host.view(torch.uint8)
    scratch = torch.empty(int(L.t3d_fill_holes_scratch_bytes(1, H, W)) // 4, dtype=torch.int32, device=dev)
    main = torch.cuda.current_stream()
    s_in, s_out = _copy_stream_pair(dev)
    start = torch.cuda.Event()
    start.record(main)
    s_in.wait_event(start)
    s_out.wait_event(start)
    bounds = [(a, min(Z, a + chunk_planes)) for a in range(0, Z, chunk_planes)]
    n_chunks = len(bounds)

    def finish(c):  # gap fill (or copy) + unpack + download of chunk c; needs chunk c+1 packed when it exists
        a, b = bounds[c]
        if close_ends:
            lo = bits[a - 1] if a > 0 else None
            hi = bits[b] if b < Z else None
            check(L.t3d_gap_fill(_p(bits[a]), _p(out_bits[a]), _p(lo), _p(hi), b - a, H, W, _p(counts[a:]), _stream()), "t3d_gap_fill")
        check(L.t3d_unpack_bits(_p(out_bits[a]), b - a, H, W, _p(out_u8[a]), _stream()), "t3d_unpack_bits")
        ev = torch.cuda.Event()
        ev.record(main)
        s_out.wait_event(ev)
        with torch.cuda.stream(s_out):
            host_u8[a:b].copy_(out_u8[a:b], non_blocking=True)

    for c, (a, b) in enumerate(bounds):
        chunk = src[a:b] if ring is None else ring.stage(source, a, b)
        with torch.cuda.stream(s_in):
            masks_dev[a:b].copy_(chunk, non_blocking=True)
            up = torch.cuda.Event()
            up.record(s_in)
            if ring is not None:
                ring.release(s_in)
        main.wait_event(up)
        dst = bits if close_ends else out_bits
        check(L.t3d_pack_masks(_p(masks_dev[a]), b - a, H, W, int(threshold), _p(dst[a]), _stream()), "t3d_pack_masks")
        if close_ends:
            if a == 0:
                check(L.t3d_fill_holes_2d(_p(bits[0]), 1, 0, H, W, _p(scratch), _stream()), "t3d_fill_holes_2d")
            if b == Z and Z > 1:
                check(L.t3d_fill_holes_2d(_p(bits[Z - 1]), 1, 0, H, W, _p(scratch), _stream()), "t3d_fill_holes_2d")
        if c > 0:
            finish(c - 1)
    finish(n_chunks - 1)
    done = torch.cuda.Event()
    done.record(s_out)
    main.wait_event(done)
    main.synchronize()
    dv = DeviceVolume(out_bits, Z, H, W, counts if close_ends else None)
    return dv, host.numpy()


def volume_from_host(voxel_data: np.ndarray) -> DeviceVolume:
    dv = volumes.lookup(voxel_data)
    if dv is not None:
        return dv
    arr = np.asarray(voxel_data)
    if arr.ndim != 3:
        raise ValueError("voxel data must be (Z,H,W)")
    return pack(upload_u8(_as_stack(arr)), 1)


# ----------------------------------------------------------------------------------------------------------
# VoxelProcessor stages
# ----------------------------------------------------------------------------------------------------------
def close_volume_ends(dv: DeviceVolume, lo_plane: Optional[torch.Tensor] = None,
                      hi_plane: Optional[torch.Tensor] = None, fill_first: bool = True,
                      fill_last: bool = True, in_place: bool = True) -> DeviceVolume:
    """voxel_processor.py:56-77.  lo/hi planes and fill_* flags exist for z-slab sharding."""
    L = _L()
    Z, H, W = dv.shape
    wpr = words_per_row(W)
    bits = dv.bits if in_place else dv.bits.clone()
    planes: List[int] = []
    if fill_first:
        planes.append(0)
    if fill_last and (Z - 1) not in planes:
        planes.append(Z - 1)
    if planes:
        scratch = torch.empty(int(L.t3d_fill_holes_scratch_bytes(len(planes), H, W)) // 4, dtype=torch.int32,
                              device=bits.device)
        if len(planes) == 2:
            check(L.t3d_fill_holes_2d(_p(bits), 2, (Z - 1) * H * wpr, H, W, _p(scratch), _stream()), "t3d_fill_holes_2d")
        else:
            check(L.t3d_fill_holes_2d(_p(bits[planes[0]]), 1, 0, H, W, _p(scratch), _stream()), "t3d_fill_holes_2d")
    out = torch.empty_like(bits)
    counts = torch.empty(Z, dtype=torch.int64, device=bits.device)
    check(L.t3d_gap_fill(_p(bits), _p(out), _p(lo_plane), _p(hi_plane), Z, H, W, _p(counts), _stream()), "t3d_gap_fill")
    return DeviceVolume(out, Z, H, W, counts)


def morph_stages(iterations: int, create_manifold: bool) -> List[bool]:
    """Stage list (True = erosion) of smooth_voxel_data, voxel_processor.py:86-91.  Closing is idempotent
    (SURVEY.md V4), so iterations >= 1 closings collapse to one."""
    stages: List[bool] = []
    if create_manifold:
        stages += [True, False]          # binary_opening = dilate(erode(x))
    if iterations >= 1:
        stages += [False, True]          # binary_closing = erode(dilate(x))
    return stages


def morph(dv: DeviceVolume, stages: Sequence[bool], want_counts: bool = True) -> DeviceVolume:
    L = _L()
    Z, H, W = dv.shape
    stages = list(stages)
    if not stages:
        return DeviceVolume(dv.bits.clone(), Z, H, W, None)
    if len(stages) > 32:
        raise ValueError("at most 32 morphology stages per call")
    mask = 0
    for s, er in enumerate(stages):
        if er:
            mask |= 1 << s
    out = torch.empty_like(dv.bits)
    counts = torch.empty(Z, dtype=torch.int64, device=out.device) if want_counts else None
    nb = int(L.t3d_morph_scratch_bytes(Z, H, W, len(stages)))
    scratch = torch.empty(nb // 4, dtype=torch.int32, device=out.device) if nb else None
    check(L.t3d_morph(_p(dv.bits), _p(out), Z, H, W, len(stages), mask, _p(counts), _p(scratch), _stream()), "t3d_morph")
    return DeviceVolume(out, Z, H, W, counts)


def smooth(dv: DeviceVolume, iterations: int = 3, create_manifold: bool = True) -> DeviceVolume:
    return morph(dv, morph_stages(iterations, create_manifold))


# ----------------------------------------------------------------------------------------------------------
# SurfaceExtractor stages
# ----------------------------------------------------------------------------------------------------------
def z_map_arrays(slice_depths, add_padding: bool) -> Tuple[np.ndarray, np.ndarray]:
    """cumulative / adjusted depths of _apply_variable_slice_depths (surface_extractor.py:84-95), host float64."""
    sd = np.asarray(slice_depths, dtype=np.float64)
    if len(sd) == 0:
        return np.zeros(0), np.zeros(0)
    adj = np.concatenate([[sd[0]], sd, [sd[-1]]]) if add_padding else sd
    cum = np.cumsum(np.concatenate([[0], adj]))
    return cum, adj


def z_map_value(plane_unpadded: float, cum: np.ndarray, adj: np.ndarray) -> np.float32:
    """float32 z coordinate the vertex transform gives to a vertex lying exactly on un-padded plane index `plane`
    (surface_extractor.py:98-113; same arithmetic as the kernel and SURVEY.md V8)."""
    z = np.float32(plane_unpadded)
    if len(cum) == 0:
        return z
    if z < 0:
        return np.float32(0)
    if z >= len(cum) - 1:
        return np.float32(cum[-1])
    lo = int(np.floor(z))
    fr = np.float32(z - np.float32(lo))
    return np.float32(cum[lo] + np.float64(fr) * adj[min(lo, len(adj) - 1)])


def zkey_bits(slice_depths, add_padding: bool, n_planes: int, z_offset: int = 0, shift: int = 1) -> int:
    """Bits needed for `float key(z) - float key(z of the layer's lower plane)` over the cube layers of a sign volume of
    n_planes planes: the bound t3d_mesh_canonicalize_structured_dev uses to shorten its radix sort (32 = no bound)."""
    cum, adj = z_map_arrays(slice_depths, add_padding)
    if len(cum) == 0:
        return 32
    z = np.array([z_map_value(k + z_offset - shift, cum, adj) for k in range(n_planes + 1)], dtype=np.float32)
    if (z < 0).any() or (np.diff(z) < 0).any():
        return 32
    span = int(np.diff(z.view(np.uint32).astype(np.int64)).max()) if len(z) > 1 else 0
    nb = max(1, span.bit_length())
    return nb if nb < 31 else 32


EXC_CAP = 1 << 20  # list capacity of the lean field-sign kernel (words needing the exact float64 evaluation); the same
                   # constant as EXC_CAP in csrc/t3d_pipeline.cu, so the staged and the fused path switch over at the same input


def field_sign(dv: DeviceVolume, pad: int, lean: bool = False):
    """Sign volume of the marched field.  lean=True uses the two-kernel variant and additionally returns the device
    counter of recorded exception words: above EXC_CAP the caller must call again with lean=False."""
    Z, H, W = dv.shape
    Zp, Hp, Wp = Z + 2 * pad, H + 2 * pad, W + 2 * pad
    dev = dv.bits.device
    sign = torch.empty((Zp, Hp, words_per_row(Wp)), dtype=torch.int32, device=dev)
    n_exact = torch.empty(1, dtype=torch.int64, device=dev)
    if not lean:
        check(_L().t3d_field_sign(_p(dv.bits), Z, H, W, pad, _W3_C, _p(sign), _p(n_exact), _stream()), "t3d_field_sign")
        return sign, (Zp, Hp, Wp), n_exact
    exc = torch.empty(EXC_CAP, dtype=torch.int64, device=dev)
    n_exc = torch.empty(1, dtype=torch.int64, device=dev)
    check(_L().t3d_field_sign_lean(_p(dv.bits), Z, H, W, pad, _W3_C, _p(sign), _p(n_exact), _p(exc), EXC_CAP, _p(n_exc),
                                   _stream()), "t3d_field_sign_lean")
    return sign, (Zp, Hp, Wp), n_exact, n_exc


def exclusive_scan_u32(x: torch.Tensor, n: int, n_arrays: int, out_u64: bool = False, popcount_input: bool = False,
                       totals: Optional[torch.Tensor] = None):
    """Exclusive scans of the n_arrays arrays of n elements stored back to back in x -> (scans, device int64 totals).
    totals: where the n_arrays totals go (a slice of a device sizes block); a new tensor if None."""
    L = _L()
    ws = torch.empty(int(L.t3d_scan_workspace_bytes(n, n_arrays)) // 8 + 1, dtype=torch.int64, device=x.device)
    if totals is None:
        totals = torch.empty(n_arrays, dtype=torch.int64, device=x.device)
    out = torch.empty(n * n_arrays, dtype=torch.int64 if out_u64 else torch.int32, device=x.device)
    check(L.t3d_exclusive_scan_u32_dev(_p(x), _p(out), n, n, n_arrays, 1 if out_u64 else 0, 1 if popcount_input else 0, None,
                                       _p(totals), _p(ws), _stream()),
          "t3d_exclusive_scan_u32_dev")
    return out, totals


def extract_surface(dv: DeviceVolume, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold: bool = True,
                    add_padding: bool = True, canonical: Optional[bool] = None, mark=None,
                    z_begin: int = 0, z_end: int = -1, z_offset: int = 0, field: Optional[torch.Tensor] = None,
                    level: float = 0.5, normals: bool = False) -> DeviceMesh:
    """surface_extractor.py:43-68 on the device.  Raises RuntimeError/ValueError where skimage would.

    z_begin / z_end / z_offset: z-slab sharding (sharded.py): owned planes of the local sign volume and the global
    padded plane index of local padded plane 0.
    normals=True: the mesh keeps what the normals kernel reads, and `mesh.normals` is the device float32 (V', 3) array of
    field-gradient normals (computed on first access, DESIGN.md §2)."""
    L = _L()
    mark = mark or (lambda _n: None)
    if field is not None:     # march a dense float32 field (SDF path): dv is ignored
        Z, H, W = (int(v) for v in field.shape)
        sbits = torch.empty((Z, H, words_per_row(W)), dtype=torch.int32, device=field.device)
        check(L.t3d_sign_from_f32(_p(field), Z, H, W, float(level), _p(sbits), _stream()), "t3d_sign_from_f32")
        dv, manifold = DeviceVolume(sbits, Z, H, W), False
    Z, H, W = dv.shape
    pad = 1 if (manifold and add_padding) else 0
    gaussian = 1 if manifold else 0
    if Z + 2 * pad < 2 or H + 2 * pad < 2 or W + 2 * pad < 2:
        raise ValueError("Input array must be at least 2x2x2.")
    dev = dv.bits.device
    # host-side constants go up before the first synchronisation point
    cum, adj = z_map_arrays(slice_depths, add_padding)
    n_cum = len(cum)
    cum_d = torch.from_numpy(cum).to(dev, non_blocking=True) if n_cum else None
    adj_d = torch.from_numpy(adj).to(dev, non_blocking=True) if n_cum else None
    n_exc_t = None
    if gaussian:
        sign, (Zs, Hs, Ws), n_exact_t, n_exc_t = field_sign(dv, pad, lean=True)
    else:
        sign, (Zs, Hs, Ws), n_exact_t = dv.bits, (Z, H, W), None
    mark("field_sign")
    n_chunks = int(L.t3d_mc_num_chunks(Zs, Hs, Ws))
    ballots = torch.empty(n_chunks, dtype=torch.int32, device=dev)
    # device sizes block {n_active, n_x, n_y, n_z, n_t} (include/t3d.h): the two scans write their totals into it
    sizes = torch.empty(5, dtype=torch.int64, device=dev)

    def flag_and_rank():
        check(L.t3d_mc_flags(_p(sign), Zs, Hs, Ws, z_begin, z_end, _p(ballots), _stream()), "t3d_mc_flags")
        return exclusive_scan_u32(ballots, n_chunks, 1, popcount_input=True, totals=sizes[:1])[0]

    chunkbase = flag_and_rank()
    mark("mc_flags")
    if n_exc_t is not None:
        n_active, n_exc = (int(v) for v in torch.cat([sizes[:1], n_exc_t]).cpu().tolist())
        if n_exc > EXC_CAP:  # too many isolated voxels for the exception list: robust single-kernel variant
            sign, _, n_exact_t = field_sign(dv, pad, lean=False)
            chunkbase = flag_and_rank()
            n_active = int(sizes[0].cpu().item())
    else:
        n_active = int(sizes[0].cpu().item())
    if n_active == 0:
        # skimage: ValueError (level outside the data range) or RuntimeError (no surface)
        raise RuntimeError("No surface found at the given iso value.")
    aw_idx = torch.empty(n_active, dtype=torch.int32, device=dev)
    aw_cnt = torch.empty(4 * n_active, dtype=torch.int32, device=dev)
    n_amb = torch.empty(1, dtype=torch.int64, device=dev)
    # what Lewiner's face / interior tests evaluate on ambiguous cubes: the dense field, or the Gaussian of the occupancy
    from ._lib import McField
    if field is not None:
        mcf = McField(None, Z, H, W, 0, 0, None, _p(field), float(level))
    else:
        mcf = McField(_p(dv.bits), Z, H, W, pad, gaussian, ctypes.cast(_W3_C, ctypes.c_void_p), None, 0.5)
    mcf_p = ctypes.cast(ctypes.pointer(mcf), ctypes.c_void_p)
    check(L.t3d_mc_words_dev(_p(sign), Zs, Hs, Ws, z_begin, z_end, _p(ballots), _p(chunkbase), n_active, _p(sizes), _p(aw_idx),
                             _p(aw_cnt), _p(n_amb), mcf_p, _stream()), "t3d_mc_words_dev")
    aw_base, _ = exclusive_scan_u32(aw_cnt, n_active, 4, totals=sizes[1:])
    mark("mc_words")
    tail = torch.cat([sizes[1:], n_amb, n_exact_t if n_exact_t is not None else torch.zeros_like(n_amb)]).cpu().tolist()
    nX, nY, nZ, nT, n_ambiguous, n_exact = (int(v) for v in tail)
    V = nX + nY + nZ
    if nT == 0 or V == 0:
        raise RuntimeError("No surface found at the given iso value.")
    if V >= 2 ** 31 or nT >= 2 ** 31:
        raise T3DError("mesh too large for one device (V=%d, F=%d)" % (V, nT))
    verts = torch.empty((V, 3), dtype=torch.float32, device=dev)
    faces = torch.empty((nT, 3), dtype=torch.int32, device=dev)
    vkeys = torch.empty(V, dtype=torch.int64, device=dev)
    strong = isinstance(mm_per_pixel_y, np.floating) or isinstance(mm_per_pixel_x, np.floating)
    check(L.t3d_mc_emit_dev(_p(sign), Zs, Hs, Ws, z_begin, z_end, _p(ballots), _p(chunkbase), _p(aw_idx), _p(aw_base), n_active,
                            _p(sizes), V, nT, _p(vkeys), _p(faces), 3, mcf_p, _stream()), "t3d_mc_emit_dev")
    mark("mc_emit")
    occ = None if field is not None else dv.bits     # the vertex and normal kernels read the dense field if one is given
    unpad = 1 if manifold else 0
    check(L.t3d_mc_vertices_dev(_p(occ), Z, H, W, pad, gaussian, _W3_C, _p(field), float(level), _p(vkeys), _p(sizes), V, unpad,
                                z_offset, _p(cum_d), _p(adj_d), n_cum, float(mm_per_pixel_y), float(mm_per_pixel_x),
                                1 if strong else 0, 7, _p(verts), _stream()), "t3d_mc_vertices_dev")
    mark("mc_vertices")
    src = None
    if normals:
        src = {"occ": occ, "field": field, "dims": (Z, H, W), "pad": pad, "gaussian": gaussian, "level": float(level), "vkeys": vkeys,
               "sizes": sizes, "unpad": unpad, "z_offset": z_offset, "adj": adj_d, "n_cum": n_cum,
               "mm": (float(mm_per_pixel_y), float(mm_per_pixel_x))}
    keep = {} if normals else None
    if canonical is None:
        canonical = manifold or field is not None
    if not canonical:
        m = DeviceMesh(verts, faces, n_ambiguous, n_exact)
        m.normal_src = src
        return m
    # structured ordering (no global sort: x-edge vertices are in place, y-edge vertices ranked per row gap, z-edge vertices
    # ordered per cube layer); the generic sort-based path only if its device-side order check fails.  "async": capacity-sized
    # arrays, the sizes stay on the device until the mesh is resolved.
    sync = canonical != "async"
    res = canonicalize_structured(verts, vkeys, faces, sizes, nZ, (Zs, Hs, Ws), chunkbase, aw_base, n_active, z_offset, unpad,
                                  cum_d, adj_d, n_cum, zkey_bits(slice_depths, add_padding, Zs, z_offset, unpad), sync=sync, keep=keep)
    if res is None:
        res = canonicalize(verts, faces, sync=sync, fast=True, keep=keep)
    mark("canonicalize")
    m = DeviceMesh(res[0], res[1], n_ambiguous, n_exact, counts_dev=None if sync else res[2])
    if not sync:
        m.raw = (verts, faces)
    m.n_active, m.n_raw, m.n_z = n_active, (V, nT), nZ
    if normals:
        m.normal_src, m.canon_map = src, keep["map"]
    return m


def canonical_map(ws: torch.Tensor, kind: int, V: int, F: int, cap_z: int = 0, cap_g0: int = 0, Zs: int = 0):
    """(newid, perm, scratch, dup flag or None, workspace) of a finished canonicalisation: device addresses of its raw ->
    canonical map inside workspace `ws` (t3d_canonical_map_offsets; kind 0 generic, 1 fast, 2 structured).  The tuple
    keeps the workspace alive."""
    off = (ctypes.c_int64 * 4)()
    check(_L().t3d_canonical_map_offsets(int(kind), int(V), int(F), int(cap_z), int(cap_g0), int(Zs), off), "t3d_canonical_map_offsets")
    base = ws.data_ptr()
    return (base + off[0], base + off[1], base + off[2], base + off[3] if off[3] >= 0 else None, ws)


def mesh_normals(mesh: DeviceMesh) -> torch.Tensor:
    """Field-gradient normals of a mesh from extract_surface(normals=True): one launch of t3d_mc_normals_dev (plus its tie pass
    when the canonicalisation may have merged vertices), rows in the mesh's vertex order."""
    src = mesh.normal_src
    n_rows = int(mesh.verts.shape[0])          # (resolves an asynchronous canonicalisation and its map first)
    out = torch.empty((n_rows, 3), dtype=torch.float32, device=src["vkeys"].device)
    newid = perm = dup = scratch = None
    if mesh.canon_map is not None:
        newid, perm, scratch, dup = (None if a is None else ctypes.c_void_p(a) for a in mesh.canon_map[:4])
    Z, H, W = src["dims"]
    check(_L().t3d_mc_normals_dev(_p(src["occ"]), Z, H, W, src["pad"], src["gaussian"], _W3_C, _p(src["field"]), src["level"],
                                  _p(src["vkeys"]), _p(src["sizes"]), int(src["vkeys"].shape[0]), src["unpad"], src["z_offset"],
                                  _p(src["adj"]), src["n_cum"], src["mm"][0], src["mm"][1], newid, perm, dup, scratch, _p(out),
                                  _stream()), "t3d_mc_normals_dev")
    return out


def canonicalize(verts: torch.Tensor, faces_i32: torch.Tensor, faces_i64: bool = True, sync: bool = True,
                 fast: bool = False, keep: Optional[dict] = None):
    """_ensure_manifold_mesh (surface_extractor.py:115-126) on the device.

    fast=True (meshes in t3d_mc_emit_dev's vertex order only): one stable 64-bit (z,y)-key sort, verified on the device;
    if the verification fails the general three-key path runs instead (sync=True) or the caller must do so
    (sync=False: returns capacity-sized arrays and the device tensor (V', F', unverified-flag)).
    keep (a dict): receives keep["map"] = canonical_map(...) of the canonicalisation that produced the result."""
    L = _L()
    V, F = int(verts.shape[0]), int(faces_i32.shape[0])
    dev = verts.device
    vout = torch.empty((V, 3), dtype=torch.float32, device=dev)
    fout = torch.empty((F, 3), dtype=torch.int64 if faces_i64 else torch.int32, device=dev)
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    f64, f32 = (_p(fout), None) if faces_i64 else (None, _p(fout))
    if fast:
        ws = torch.empty(int(L.t3d_canonicalize_fast_workspace_bytes(V, F)) // 8 + 1, dtype=torch.int64, device=dev)
        check(L.t3d_mesh_canonicalize_fast_dev(_p(verts), V, None, _p(faces_i32), F, None, _p(vout), f64, f32, _p(counts), _p(ws),
                                               _stream()), "t3d_mesh_canonicalize_fast_dev")
    else:
        ws = torch.empty(int(L.t3d_canonicalize_workspace_bytes(V, F)) // 8 + 1, dtype=torch.int64, device=dev)
        check(L.t3d_mesh_canonicalize(_p(verts), V, _p(faces_i32), F, _p(vout), f64, f32, _p(counts), _p(ws), _stream()),
              "t3d_mesh_canonicalize")
    if keep is not None:
        keep["map"] = canonical_map(ws, 1 if fast else 0, V, F)
    if not sync:
        return vout, fout, counts
    v2, f2, bad = (int(c) for c in counts.cpu().tolist())
    if bad:
        return canonicalize(verts, faces_i32, faces_i64, True, False, keep=keep)
    return vout[:v2], fout[:f2]


def canonicalize_structured(verts, vkeys, faces_i32, sizes, n_z, sign_dims, chunkbase, aw_base, aw_stride, z_offset, unpad_shift,
                            cum_d, adj_d, n_cum, zkey_bits_, sync: bool = True, keep: Optional[dict] = None):
    """_ensure_manifold_mesh for a mesh straight out of t3d_mc_emit_dev (t3d_mesh_canonicalize_structured_dev); `sizes` is the
    extraction's device sizes block, n_z its z-edge vertex count.
    sync=True: returns (verts, int64 faces) or None when the structured order could not be verified (the caller then sorts
    generically); the clamp group (vertices under slice 0) is provisioned on a second attempt when the first one reports it.
    sync=False: one attempt, returns capacity-sized (verts, faces, device counts (V', F', unverified flag)).
    keep (a dict): receives keep["map"] = canonical_map(...) of the last attempt."""
    L = _L()
    V, nT = int(verts.shape[0]), int(faces_i32.shape[0])
    Zs, Hs, Ws = sign_dims
    dev = verts.device
    vout = torch.empty((V, 3), dtype=torch.float32, device=dev)
    fout = torch.empty((nT, 3), dtype=torch.int64, device=dev)
    counts = torch.zeros(4, dtype=torch.int64, device=dev)
    cap_z, cap_g0 = max(n_z, 1), 0
    for _attempt in range(2):
        ws = torch.zeros(int(L.t3d_canonicalize_structured_workspace_bytes(V, nT, cap_z, cap_g0, Zs)) // 8 + 1, dtype=torch.int64, device=dev)
        check(L.t3d_mesh_canonicalize_structured_dev(
            _p(verts), _p(vkeys), V, _p(sizes), None, Zs, Hs, Ws, _p(chunkbase), _p(aw_base), int(aw_stride), int(z_offset),
            int(unpad_shift), _p(cum_d), _p(adj_d), int(n_cum), int(zkey_bits_), cap_z, cap_g0, _p(faces_i32), nT, None,
            _p(vout), _p(fout), None, _p(counts), _p(counts[3:]), _p(ws), 3, _stream()), "t3d_mesh_canonicalize_structured_dev")
        if keep is not None:
            keep["map"] = canonical_map(ws, 2, V, nT, cap_z, cap_g0, Zs)
        if not sync:
            return vout, fout, counts[:3]
        v2, f2, bad, n_g0 = (int(c) for c in counts.cpu().tolist())
        if not bad:
            return vout[:v2], fout[:f2]
        if n_g0 > cap_g0:
            cap_g0 = n_g0 + 16
            continue
        break
    return None


def mesh_measure_async(verts: torch.Tensor, faces: torch.Tensor) -> torch.Tensor:
    """Device tensor {signed volume, area} (float64), no synchronisation."""
    L = _L()
    dev = verts.device
    ws = torch.empty(int(L.t3d_mesh_measure_workspace_bytes()) // 8, dtype=torch.float64, device=dev)
    out = torch.empty(2, dtype=torch.float64, device=dev)
    verts = verts.contiguous()
    faces = faces.contiguous()
    check(L.t3d_mesh_measure_dev(_p(verts), _p(faces), int(faces.shape[0]), None, 1 if faces.dtype == torch.int64 else 0, _p(out),
                                 _p(ws), _stream()), "t3d_mesh_measure_dev")
    return out


def mesh_measure(verts: torch.Tensor, faces: torch.Tensor) -> Tuple[float, float]:
    v, a = mesh_measure_async(verts, faces).cpu().tolist()
    return float(v), float(a)


def mesh_from_host(vertices: np.ndarray, faces: np.ndarray) -> DeviceMesh:
    m = meshes.lookup(vertices)
    if m is not None and meshes.lookup(faces) is m:
        return m
    dev = _require_cuda()
    f = np.ascontiguousarray(faces)
    if f.dtype not in (np.int32, np.int64):
        f = f.astype(np.int64)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)  # read-only ndarray -> tensor (we only read it)
        v = torch.from_numpy(np.ascontiguousarray(vertices, dtype=np.float32)).to(dev)
        return DeviceMesh(v, torch.from_numpy(f).to(dev))


# ----------------------------------------------------------------------------------------------------------
# point cloud (voxel_processor.py:99-127)
# ----------------------------------------------------------------------------------------------------------
def point_cloud(dv: DeviceVolume, mm_per_pixel_x, mm_per_pixel_y, slice_depths, subsample_factor: int = 1) -> np.ndarray:
    L = _L()
    Z, H, W = dv.shape
    dev = dv.bits.device
    rows = Z * H
    rc = torch.empty(rows, dtype=torch.int32, device=dev)
    check(L.t3d_row_popcounts(_p(dv.bits), Z, H, W, _p(rc), _stream()), "t3d_row_popcounts")
    base, total = exclusive_scan_u32(rc, rows, 1, out_u64=True)
    n = int(total.cpu().item())
    sub = subsample_factor if subsample_factor > 1 else 1
    n_out = (n + sub - 1) // sub
    sd = np.asarray(slice_depths, dtype=np.float64)
    cum = np.cumsum(np.concatenate([[0], sd]))
    zc = np.empty(Z, dtype=np.float64)
    k = min(Z, len(sd))
    zc[:k] = cum[:k] + sd[:k] / 2          # centre of slice (voxel_processor.py:116-117)
    zc[k:] = cum[-1]                       # (:118-119)
    out = torch.empty((n_out, 3), dtype=torch.float64, device=dev)
    if n_out:
        check(L.t3d_point_cloud_emit(_p(dv.bits), Z, H, W, _p(base), sub, _p(torch.from_numpy(zc).to(dev)),
                                     float(mm_per_pixel_y), float(mm_per_pixel_x), _p(out), _stream()),
              "t3d_point_cloud_emit")
    return out.cpu().numpy()
