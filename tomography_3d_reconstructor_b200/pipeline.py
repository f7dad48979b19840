"""Whole-job pipeline on device-resident inputs: uint8 mask stack -> voxel grid -> smoothing -> mesh + volumes.

This is the order tomography_3d_reconstruction.py runs the hot path in (create_voxel_data :88-100, calculate_volume
:102-118, smooth + extract + mesh volume :120-140, surface area :207-223, analyze :225-229), run once per step
instead of the orchestrator's 5x smooth / 4x extract on identical inputs (SURVEY.md 3.1).
"""
from __future__ import annotations

from typing import Callable, Dict, Optional

import numpy as np
import torch

from . import engine


def slice_depths(total_depth_mm: float, side_0: int, side_1: int, side_2: int) -> np.ndarray:
    """voxel_processor.py:129-163 (host scalars)."""
    total = side_0 + side_1 + side_2
    if side_1 == 0 or total == 0:
        return np.array([]) if total == 0 else np.full(total, total_depth_mm / total)
    d1 = total_depth_mm / side_1
    d02 = 2 * d1
    d0 = d02 / side_0 if side_0 > 0 else 0
    d2 = d02 / side_2 if side_2 > 0 else 0
    return np.array([d0] * side_0 + [d1] * side_1 + [d2] * side_2)


def volume_weights(mm_x: float, mm_y: float, depths: np.ndarray) -> np.ndarray:
    """Per-slice voxel volume `mm_x * mm_y * depth[z]` exactly as volume_calculator.py:31-33 forms it."""
    return (mm_x * mm_y) * np.asarray(depths, dtype=np.float64)


def variable_depth_volume(counts: np.ndarray, mm_x: float, mm_y: float, depths: np.ndarray, weights: np.ndarray = None) -> float:
    """volume_calculator.py:23-35 on exact per-slice counts, same float64 order.  `weights` = volume_weights(...) cached
    by the caller (the fused plans call this between two steps, with the GPU idle)."""
    if len(depths) == 0:
        return 0.0
    n = min(len(counts), len(depths))
    if n == 0:
        return 0.0
    if weights is None:
        weights = volume_weights(mm_x, mm_y, depths)
    # the reference's loop `total += count[z] * (mm_x * mm_y * depth[z])`, vectorised without changing a bit:
    # the products are the same float64 operations and np.cumsum accumulates strictly left to right
    prod = np.asarray(counts[:n]).astype(np.float64) * weights[:n]
    return float(np.cumsum(prod)[-1])


def reconstruct(masks_u8: torch.Tensor, threshold: int, side_counts, total_depth_mm: float, x_length_mm: float,
                y_length_mm: float, iterations: int = 3, close_ends: bool = True, add_padding: bool = True,
                mark: Optional[Callable[[str], None]] = None, normals: bool = False) -> Dict:
    """masks_u8: CUDA uint8 (Z,H,W).  Returns the device mesh and the host scalars of analyze_object_properties.

    `mark(name)` is called after each stage has been enqueued (bench.py records CUDA events there).
    normals=True: also "normals", the device float32 (V', 3) field-gradient normals of the mesh (DESIGN.md §2)."""
    mark = mark or (lambda _n: None)
    Z, H, W = (int(s) for s in masks_u8.shape)
    mm_x, mm_y = x_length_mm / W, y_length_mm / H
    depths = slice_depths(total_depth_mm, *side_counts)

    dv = engine.pack_and_close(masks_u8, threshold, close_ends)
    mark("pack_close")
    # bounding box of the raw grid: off the critical path
    main = torch.cuda.current_stream()
    side = engine.side_stream(masks_u8.device)
    ready = torch.cuda.Event()
    ready.record(main)
    with torch.cuda.stream(side):
        side.wait_event(ready)
        bbox_t = dv.bbox_tensor()
        bbox_done = torch.cuda.Event()
        bbox_done.record(side)
    sm = engine.smooth(dv, iterations, True)
    mark("smooth")
    mesh = engine.extract_surface(sm, depths, mm_y, mm_x, True, add_padding, canonical="async", mark=mark, normals=normals)
    # measures on the emitted (pre-canonical) mesh: merging exact duplicates and dropping zero-area faces changes
    # neither the signed volume nor the area, and it removes a dependency on the canonical sizes
    raw_verts, raw_faces = mesh.raw
    meas = engine.mesh_measure_async(raw_verts, raw_faces)
    mark("measure")
    main.wait_event(bbox_done)
    # one device->host copy for every scalar result of the step
    Zc = dv.Z
    packed = torch.cat([mesh.counts_dev, meas.view(torch.int64), dv.counts_tensor(), sm.counts_tensor(),
                        bbox_t.to(torch.int64)]).cpu()
    mark("stats")
    mesh.set_sizes(int(packed[0]), int(packed[1]), int(packed[2]))
    signed_volume, area = (float(x) for x in packed[3:5].view(torch.float64).tolist())
    mesh._measures = (signed_volume, area)
    raw_counts = packed[5:5 + Zc].numpy().astype(np.int64)
    sm_counts = packed[5 + Zc:5 + 2 * Zc].numpy().astype(np.int64)
    bb = tuple(int(x) for x in packed[5 + 2 * Zc:].tolist())
    dv.set_host_stats(raw_counts, bb)
    sm.set_host_stats(sm_counts, None)
    bbox = dv.bbox()
    out = {
        "mesh": mesh,
        "voxel_volume_mm3": variable_depth_volume(raw_counts, mm_x, mm_y, depths),
        "processed_voxel_volume_mm3": variable_depth_volume(sm_counts, mm_x, mm_y, depths),
        "mesh_volume_mm3": abs(signed_volume),
        "surface_area_mm2": area,
        "bbox_index": bbox,
        "active_voxels": int(raw_counts.sum()),
        "slice_depths": depths,
    }
    if normals:
        out["normals"] = mesh.normals
    return out


def sdf_sampling(depths: np.ndarray, mm_y: float, mm_x: float):
    """Voxel pitch (z, y, x) in mm used for the distance transform: the mean slice depth along z (the separable transform
    needs one pitch per axis; the z coordinates of the vertices still go through the exact variable-depth map)."""
    dz = float(np.mean(depths)) if len(depths) else 1.0
    return (dz if dz > 0 else 1.0, float(mm_y), float(mm_x))


def reconstruct_sdf(masks_u8: torch.Tensor, threshold: int, side_counts, total_depth_mm: float, x_length_mm: float,
                    y_length_mm: float, iterations: int = 3, close_ends: bool = True, level: float = 0.0,
                    sampling=None) -> Dict:
    """SDF variant of reconstruct() (BASELINE configs 3/4; additive, SURVEY.md 8a-16): voxel grid -> smoothing -> exact
    signed Euclidean distance (mm, positive inside) -> marching cubes on the distance field at `level` -> mesh + volumes.
    Returns reconstruct()'s dict plus "sdf" (float32 CUDA tensor)."""
    from . import edt
    Z, H, W = (int(s) for s in masks_u8.shape)
    mm_x, mm_y = x_length_mm / W, y_length_mm / H
    depths = slice_depths(total_depth_mm, *side_counts)
    dv = engine.pack_and_close(masks_u8, threshold, close_ends)
    sm = engine.smooth(dv, iterations, True)
    sdf = edt.signed_distance(sm, sampling or sdf_sampling(depths, mm_y, mm_x))
    mesh = engine.extract_surface(None, depths, mm_y, mm_x, False, False, field=sdf, level=level)
    signed_volume, area = mesh.measures()
    raw_counts, sm_counts = dv.slice_counts(), sm.slice_counts()
    return {
        "mesh": mesh, "sdf": sdf,
        "voxel_volume_mm3": variable_depth_volume(raw_counts, mm_x, mm_y, depths),
        "processed_voxel_volume_mm3": variable_depth_volume(sm_counts, mm_x, mm_y, depths),
        "mesh_volume_mm3": abs(signed_volume), "surface_area_mm2": area, "bbox_index": dv.bbox(),
        "active_voxels": int(raw_counts.sum()), "slice_depths": depths,
    }


# ----------------------------------------------------------------------------------------------------------------
# fused path: the whole step as ONE enqueue (t3d_reconstruct), captured in a CUDA graph
# ----------------------------------------------------------------------------------------------------------------
R_NACTIVE, R_NX, R_NY, R_NZ, R_NT, R_VCANON, R_FCANON, R_UNVERIFIED, R_OVERFLOW = range(9)   # keep in sync with t3d_pipeline.cu
R_NAMBIGUOUS, R_NEXACT, R_VOLUME, R_AREA, R_BBOX, R_VRAW, R_NG0, R_COUNTS = 9, 10, 11, 12, 13, 16, 25, 32


class FusedPlan:
    """Buffers + (optionally) a captured CUDA graph for one problem shape.  Data-dependent sizes stay on the device;
    buffers are capacity-sized from hints (a previous run of the same input) and the result block reports overflow.
    The mesh returned by run() lives in the plan's output buffers: valid until the next run().
    normals=True: every step is followed by t3d_reconstruct_normals (in the same graph), into `self.normals`."""

    def __init__(self, shape, threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations, close_ends,
                 add_padding, caps, device, normals: bool = False):
        L = engine._L()
        self.shape = Z, H, W = tuple(int(v) for v in shape)
        self.threshold, self.close_ends, self.add_padding = int(threshold), bool(close_ends), bool(add_padding)
        self.mm_x, self.mm_y = x_length_mm / W, y_length_mm / H
        self.depths = slice_depths(total_depth_mm, *side_counts)
        self.vol_weights = volume_weights(self.mm_x, self.mm_y, self.depths)
        stages = engine.morph_stages(iterations, True)
        self.n_stages = len(stages)
        self.erode_mask = sum(1 << k for k, er in enumerate(stages) if er)
        self.caps = tuple(int(c) for c in caps)
        cum, adj = engine.z_map_arrays(self.depths, add_padding)
        self.n_cum = len(cum)
        self.zkey_bits = engine.zkey_bits(self.depths, add_padding, Z + 2 * (1 if add_padding else 0), 0, 1)
        self.cum_d = torch.from_numpy(cum).to(device) if self.n_cum else None
        self.adj_d = torch.from_numpy(adj).to(device) if self.n_cum else None
        if len(self.caps) != 5:
            raise ValueError("caps = (active words, vertices, faces, z-edge vertices, clamp group)")
        nbytes = int(L.t3d_reconstruct_workspace_bytes(Z, H, W, 1 if add_padding else 0, self.n_stages, *self.caps))
        self.ws = torch.empty(nbytes // 8 + 1, dtype=torch.int64, device=device)
        self.verts = torch.empty((self.caps[1], 3), dtype=torch.float32, device=device)
        self.faces = torch.empty((self.caps[2], 3), dtype=torch.int64, device=device)
        self.normals = torch.empty((self.caps[1], 3), dtype=torch.float32, device=device) if normals else None
        self.n_res = int(L.t3d_reconstruct_results_len(Z))
        self.res = torch.zeros(self.n_res, dtype=torch.int64, device=device)
        self.res_host = torch.zeros(self.n_res, dtype=torch.int64, pin_memory=True)
        self.res_np = self.res_host.numpy()
        self.graph, self.graph_ptr = None, None
        self.last_sizes, self.last_canon, self.last_mesh = None, None, None

    def enqueue(self, masks_u8: torch.Tensor) -> None:
        Z, H, W = self.shape
        p = engine._p
        engine.check(engine._L().t3d_reconstruct(
            p(masks_u8), Z, H, W, self.threshold, 1 if self.close_ends else 0, self.n_stages, self.erode_mask,
            1 if self.add_padding else 0, engine._W3_C, p(self.cum_d), p(self.adj_d), self.n_cum, float(self.mm_y),
            float(self.mm_x), 0, self.caps[0], self.caps[1], self.caps[2], self.caps[3], self.caps[4], self.zkey_bits, p(self.verts),
            p(self.faces), p(self.res), p(self.ws), engine._stream()), "t3d_reconstruct")
        if self.normals is not None:
            engine.check(engine._L().t3d_reconstruct_normals(
                Z, H, W, self.n_stages, self.erode_mask, 1 if self.add_padding else 0, engine._W3_C, p(self.adj_d), self.n_cum,
                float(self.mm_y), float(self.mm_x), *self.caps, p(self.res), p(self.ws), p(self.normals), engine._stream()),
                "t3d_reconstruct_normals")

    def capture(self, masks_u8: torch.Tensor) -> None:
        """Record the step for this input buffer into a CUDA graph (after one eager warm-up run)."""
        self.enqueue(masks_u8)
        torch.cuda.current_stream().synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=engine.capture_stream()):
            self.enqueue(masks_u8)
            self.res_host.copy_(self.res, non_blocking=True)      # the read-back of the result block is a node of the graph
        self.graph, self.graph_ptr = g, masks_u8.data_ptr()
        self.res_np = self.res_host.numpy()

    def launch(self, masks_u8: torch.Tensor, use_graph: bool = True) -> None:
        """Enqueue one step on the current stream (graph replay when captured for this input buffer); no synchronisation."""
        if use_graph and self.graph is not None and self.graph_ptr == masks_u8.data_ptr():
            self.graph.replay()
        else:
            self.enqueue(masks_u8)
            self.res_host.copy_(self.res, non_blocking=True)

    def run(self, masks_u8: torch.Tensor, use_graph: bool = True):
        """Returns the host result block (numpy int64 view) after one synchronisation."""
        self.launch(masks_u8, use_graph)
        torch.cuda.current_stream().synchronize()
        return self.res_np


_plans: Dict = {}
_hints: Dict = {}
_g0_caps: Dict = {}       # key -> capacity of the z-clamp group sort (survives re-learning of the other capacities)
_generic_sort: Dict = {}  # key -> True: the structured vertex ordering could not be verified on this input, use the 64-bit sort


def _tuned_caps(key, caps):
    caps = tuple(caps)
    g0 = max(caps[4], _g0_caps.get(key, 0))
    return caps[:3] + ((0, 0) if _generic_sort.get(key) else (caps[3], g0))


def _retune(key, n_g0: int, cap_g0: int) -> bool:
    """After an unverified structured ordering: provision the clamp-group sort if that was missing, else switch this
    problem to the generic 64-bit sort.  Returns True if the step should be run again."""
    if n_g0 > cap_g0:
        _g0_caps[key] = _grow(n_g0)
    else:
        _generic_sort[key] = True
    return True


def _grow(n: int) -> int:
    return int(n * 1.02) + 4096


def _caps_from(n_active: int, v_raw: int, f_raw: int, n_z: int, n_g0: int = 0):
    """Capacities (active words, vertices, faces, z-edge vertices, z-clamp group) with a small margin; the clamp group
    (vertices under slice 0, see t3d_mesh_canonicalize_structured_dev) stays unprovisioned while it is empty."""
    return _grow(n_active), _grow(v_raw), _grow(f_raw), _grow(n_z), (_grow(n_g0) if n_g0 > 0 else 0)


def plan_key(masks_u8: torch.Tensor, threshold: int, side_counts, total_depth_mm: float, x_length_mm: float,
             y_length_mm: float, iterations: int = 3, close_ends: bool = True, add_padding: bool = True, normals: bool = False):
    """Key of the fused plan / capacity hints of one problem (plans with and without normals are distinct)."""
    Z, H, W = (int(s) for s in masks_u8.shape)
    key = (Z, H, W, int(threshold), tuple(side_counts), float(total_depth_mm), float(x_length_mm), float(y_length_mm),
           int(iterations), bool(close_ends), bool(add_padding), masks_u8.device.index)
    return key + ("normals",) if normals else key


def reconstruct_fused(masks_u8: torch.Tensor, threshold: int, side_counts, total_depth_mm: float, x_length_mm: float,
                      y_length_mm: float, iterations: int = 3, close_ends: bool = True, add_padding: bool = True,
                      use_graph: bool = True, normals: bool = False) -> Dict:
    """Same contract as reconstruct(), executed as one graph launch + one device->host copy.

    The first call for a given (shape, parameters) runs the staged path to learn the mesh size; later calls reuse a
    FusedPlan.  If the input changes so much that a capacity overflows (or the fast vertex ordering cannot be
    verified) the staged path runs instead and the hints are refreshed.
    normals=True: out["normals"] is the device float32 (V', 3) array of field-gradient normals (DESIGN.md §2)."""
    Z, H, W = (int(s) for s in masks_u8.shape)
    key = plan_key(masks_u8, threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations, close_ends, add_padding,
                   normals)

    def staged():
        out = reconstruct(masks_u8, threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations, close_ends,
                          add_padding, normals=normals)
        m = out["mesh"]
        _hints[key] = _caps_from(m.n_active, *m.n_raw, m.n_z)
        return out

    if key not in _hints:
        return staged()
    caps = _tuned_caps(key, _hints[key])
    plan = _plans.get(key)
    if plan is None or any(c < h for c, h in zip(plan.caps, caps)) or (plan.caps[3] == 0) != (caps[3] == 0):
        plan = FusedPlan((Z, H, W), threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations,
                         close_ends, add_padding, caps, masks_u8.device, normals)
        _plans[key] = plan
    if use_graph and plan.graph_ptr != masks_u8.data_ptr():
        plan.capture(masks_u8)
    r = plan.run(masks_u8, use_graph)
    # (from here on: plain Python on one .tolist() of the header -- this runs between two steps, with the GPU idle)
    h = r[:R_COUNTS].tolist()
    if h[R_UNVERIFIED] and not h[R_OVERFLOW] and plan.caps[3] and _retune(key, h[R_NG0], plan.caps[4]):
        _plans.pop(key, None)
        return reconstruct_fused(masks_u8, threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations,
                                 close_ends, add_padding, use_graph, normals)
    if h[R_OVERFLOW] or h[R_UNVERIFIED] or h[R_NT] == 0:
        _plans.pop(key, None)
        _hints.pop(key, None)
        return staged()
    return _result_from_block(plan, r, h, key)


def _result_from_block(plan: "FusedPlan", r: np.ndarray, h: list, hints_key=None) -> Dict:
    """Result dict of reconstruct() from the host result block of a step that neither overflowed nor failed its order
    check (plain Python on one .tolist() of the header: this runs between two steps, with the GPU idle)."""
    Z = plan.shape[0]
    sizes = (h[R_NACTIVE], h[R_VRAW], h[R_NT], h[R_NZ], h[R_NG0])
    if sizes != plan.last_sizes:
        # every later call with a slightly larger mesh still fits thanks to the margin; refresh the hints if it grew
        if hints_key is not None and hints_key in _hints:
            _hints[hints_key] = tuple(max(a, b) for a, b in zip(_hints[hints_key], _caps_from(*sizes)))
        plan.last_sizes = sizes
    canon = (h[R_VCANON], h[R_FCANON])
    if plan.last_mesh is None or plan.last_canon != canon:
        plan.last_mesh = engine.DeviceMesh(plan.verts[:canon[0]], plan.faces[:canon[1]])
        plan.last_canon = canon
    mesh = plan.last_mesh                       # views of the plan's output buffers: valid until the next run
    mesh.n_ambiguous, mesh.n_exact = h[R_NAMBIGUOUS], h[R_NEXACT]
    vol_area = r[R_VOLUME:R_VOLUME + 2].view(np.float64).tolist()
    mesh._measures = (vol_area[0], vol_area[1])
    mesh.n_active, mesh.n_raw, mesh.n_z = sizes[0], (sizes[1], sizes[2]), sizes[3]
    # both voxel volumes in one pass: rows = raw / smoothed per-slice counts (volume_calculator.py:23-35, same order)
    counts2 = r[R_COUNTS:R_COUNTS + 2 * Z].reshape(2, Z)
    n = min(Z, len(plan.depths))
    vols = np.cumsum(counts2[:, :n].astype(np.float64) * plan.vol_weights[:n], axis=1)[:, -1].tolist() if n else [0.0, 0.0]
    bb = r[R_BBOX:R_BBOX + 3].view(np.int32).tolist()
    out = {
        "mesh": mesh,
        "voxel_volume_mm3": vols[0],
        "processed_voxel_volume_mm3": vols[1],
        "mesh_volume_mm3": abs(vol_area[0]),
        "surface_area_mm2": vol_area[1],
        "bbox_index": tuple(bb) if bb[1] >= 0 else None,
        "active_voxels": int(counts2[0].sum()),
        "slice_depths": plan.depths,
    }
    if plan.normals is not None:
        out["normals"] = plan.normals[:canon[0]]
    return out


_device_inputs: Dict = {}


def reconstruct_host(mask_images, threshold: int, side_counts, total_depth_mm: float, x_length_mm: float, y_length_mm: float,
                     iterations: int = 3, close_ends: bool = True, add_padding: bool = True, use_graph: bool = True,
                     normals: bool = False) -> Dict:
    """The whole path on HOST data, as one call: a list of (H,W) bool / uint8 masks (what ImageLoader returns,
    image_loader.py:97-109) or a (Z,H,W) array -> one host->device copy -> reconstruct_fused -> the mesh as numpy arrays
    (out["vertices"] f32 (V,3) [z,y,x] mm, out["faces"] int64 (F,3)) + the scalars of reconstruct().  bool masks:
    pass threshold=1.  The intermediate voxel grids stay on the device (the class API has to return them as arrays).
    normals=True: also out["normals"], float32 (V,3) field-gradient unit normals, row i for vertex i (DESIGN.md §2)."""
    _src, Z, H, W, _pinned = engine.mask_source(mask_images)
    dev = engine._require_cuda()
    key = ((Z, H, W), torch.cuda.current_device())
    buf = _device_inputs.get(key)
    if buf is None:                                  # persistent input buffer: keeps the captured graph valid
        buf = _device_inputs[key] = torch.empty((Z, H, W), dtype=torch.uint8, device=dev)
    # one async copy from a pinned stack; a list of pageable masks is gathered through the pinned staging ring
    engine.upload_masks(mask_images, buf)
    out = reconstruct_fused(buf, threshold, side_counts, total_depth_mm, x_length_mm, y_length_mm, iterations, close_ends,
                            add_padding, use_graph, normals)
    v, f = out["mesh"].verts.contiguous(), out["mesh"].faces.contiguous()
    hv = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
    hf = torch.empty(f.shape, dtype=f.dtype, pin_memory=True)
    hv.copy_(v, non_blocking=True)
    hf.copy_(f, non_blocking=True)
    if normals:
        n = out["normals"].contiguous()
        hn = torch.empty(n.shape, dtype=n.dtype, pin_memory=True)
        hn.copy_(n, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    out["vertices"], out["faces"] = hv.numpy(), hf.numpy()
    if normals:
        out["normals"] = hn.numpy()
    return out
