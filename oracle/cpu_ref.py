"""oracle/cpu_ref.py -- TEST INFRASTRUCTURE ONLY.

CPU restatement (numpy + scipy + oracle/mc_ref.c) of the reference's reconstruction hot path:
voxel_processor.py, surface_extractor.py and volume_calculator.py of
victorramirez952/tomography_3d_reconstructor.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module; the product package never does.

Why a restatement and not the reference itself: the reference delegates its arithmetic to
scikit-image (`scikit-image>=0.18.0`, requirements.txt:5, no exact pin), which is not installed in
this image and cannot be installed offline.  With skimage absent the reference silently degrades
(voxel_processor.py:17-24,81-82; surface_extractor.py:39-40).  Everything below that does NOT need
skimage is checked against outputs of the unmodified reference modules, stored as fixtures in
tests/golden/ (tests/test_oracle.py, tests/test_oracle_vs_reference.py).

PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures (SURVEY.md section 4), and
the two skimage entry points are restated:
  * skimage.morphology.binary_opening / binary_closing  -> scipy.ndimage.binary_erosion(structure=
    cross, border_value=True) / binary_dilation(structure=cross)   [exact by construction, scipy is
    what skimage calls]
  * skimage.measure.marching_cubes (Lewiner)             -> oracle/mc_ref.c (classic table; cubes
    whose tiling Lewiner's extra tests could change are counted, see mc_ref.c)
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Optional, Tuple

import numpy as np
from scipy import ndimage

_HERE = os.path.dirname(os.path.abspath(__file__))
_REF_DIR = os.path.join(_HERE, "_ref")
_MC_SO = os.path.join(_REF_DIR, "libmc_ref.so")


# --------------------------------------------------------------------------------------------
# build / load of the C part
# --------------------------------------------------------------------------------------------
def build(force: bool = False) -> str:
    """Compile oracle/mc_ref.c -> oracle/_ref/libmc_ref.so (gcc, no external dependencies)."""
    src = os.path.join(_HERE, "mc_ref.c")
    hdr = os.path.join(_HERE, "mc33_tables_oracle.h")      # the oracle's own tables: nothing under the product tree is included
    os.makedirs(_REF_DIR, exist_ok=True)
    if (not force and os.path.exists(_MC_SO)
            and os.path.getmtime(_MC_SO) >= max(os.path.getmtime(src), os.path.getmtime(hdr))):
        return _MC_SO
    cmd = ["gcc", "-O2", "-fPIC", "-shared", "-std=c99", "-ffp-contract=off", "-I", _HERE, src, "-o", _MC_SO, "-lm"]
    subprocess.check_call(cmd)
    return _MC_SO


_lib = None


def _mc_lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_MC_SO):
            build()
        _lib = ctypes.CDLL(_MC_SO)
        _lib.t3d_oracle_marching_cubes.restype = ctypes.c_int
        _lib.t3d_oracle_marching_cubes.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
            ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64,
            ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64),
            ctypes.POINTER(ctypes.c_int64), ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]
        _lib.t3d_oracle_resolve_cube.restype = ctypes.c_int
        _lib.t3d_oracle_resolve_cube.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib.t3d_oracle_cube_cases.restype = ctypes.c_int
        _lib.t3d_oracle_cube_cases.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_void_p]
    return _lib


# --------------------------------------------------------------------------------------------
# voxel_processor.py
# --------------------------------------------------------------------------------------------
_CROSS3 = ndimage.generate_binary_structure(3, 1)


def close_volume_ends(voxel_data: np.ndarray) -> np.ndarray:
    """voxel_processor.py:56-77 restated literally (scipy branch, :61-62 / :67-68)."""
    closed = voxel_data.copy()
    if np.any(closed[0]):
        closed[0] = ndimage.binary_fill_holes(closed[0])
    if np.any(closed[-1]):
        closed[-1] = ndimage.binary_fill_holes(closed[-1])
    for z in range(1, closed.shape[0] - 1):
        if np.any(closed[z - 1]) and np.any(closed[z + 1]):
            closed[z] = np.logical_or(closed[z], np.logical_and(closed[z - 1], closed[z + 1]))
    return closed


def close_volume_ends_stencil(voxel_data: np.ndarray) -> np.ndarray:
    """Non-recurrent form of the same function (SURVEY.md V3): what the CUDA kernels implement."""
    f = voxel_data.copy()
    f[0] = ndimage.binary_fill_holes(f[0])
    f[-1] = ndimage.binary_fill_holes(f[-1])
    out = f.copy()
    if f.shape[0] > 2:
        out[1:-1] = f[1:-1] | (f[:-2] & f[2:])
    return out


def create_voxel_data(mask_images: list, close_ends: bool = True) -> np.ndarray:
    """voxel_processor.py:36-54."""
    if not mask_images:
        raise ValueError("Load masks first, hmm.")
    vol = np.stack(mask_images, axis=0)
    if close_ends:
        vol = close_volume_ends(vol)
    return vol


def binary_erosion6(x: np.ndarray) -> np.ndarray:
    """skimage.morphology.binary_erosion default footprint: out-of-bounds counts as True."""
    return ndimage.binary_erosion(x, structure=_CROSS3, border_value=True)


def binary_dilation6(x: np.ndarray) -> np.ndarray:
    """skimage.morphology.binary_dilation default footprint: out-of-bounds counts as False."""
    return ndimage.binary_dilation(x, structure=_CROSS3)


def binary_opening6(x):
    return binary_dilation6(binary_erosion6(x))


def binary_closing6(x):
    return binary_erosion6(binary_dilation6(x))


def smooth_voxel_data(voxel_data: np.ndarray, iterations: int = 3, create_manifold: bool = True) -> np.ndarray:
    """voxel_processor.py:79-97 with skimage present (the degraded identity path :81-82 is NOT reproduced)."""
    s = voxel_data.copy()
    if create_manifold:
        s = binary_opening6(s)
    for _ in range(iterations):
        s = binary_closing6(s)
    return s


def calculate_slice_depths(total_depth_mm: float, side_0: int, side_1: int, side_2: int) -> np.ndarray:
    """voxel_processor.py:129-163."""
    total = side_0 + side_1 + side_2
    if side_1 == 0 or total == 0:
        if total == 0:
            return np.array([])
        return np.full(total, total_depth_mm / total)
    d1 = total_depth_mm / side_1
    d02 = 2 * d1
    d0 = d02 / side_0 if side_0 > 0 else 0
    d2 = d02 / side_2 if side_2 > 0 else 0
    return np.array([d0] * side_0 + [d1] * side_1 + [d2] * side_2)


def generate_point_cloud(voxel_data, mm_per_pixel_x, mm_per_pixel_y, slice_depths, subsample_factor=1):
    """voxel_processor.py:99-127 (vectorised; SURVEY.md V9 bit-exact)."""
    z, y, x = np.where(voxel_data)
    if subsample_factor > 1:
        idx = np.arange(0, len(z), subsample_factor)
        z, y, x = z[idx], y[idx], x[idx]
    cum = np.cumsum(np.concatenate([[0], slice_depths]))
    zmm = np.empty(len(z), dtype=np.float64)
    inside = z < len(slice_depths)
    zi = z[inside]
    zmm[inside] = cum[zi] + np.asarray(slice_depths)[zi] / 2
    zmm[~inside] = cum[-1]
    return np.column_stack([zmm, y * mm_per_pixel_y, x * mm_per_pixel_x])


# --------------------------------------------------------------------------------------------
# surface_extractor.py
# --------------------------------------------------------------------------------------------
def scalar_field(volume_data: np.ndarray, manifold: bool = True, add_padding: bool = True) -> np.ndarray:
    """surface_extractor.py:43-53 + skimage's float32 cast at entry: the array that is marched."""
    v = volume_data
    if manifold and add_padding:
        v = np.pad(v, 1, mode="constant", constant_values=False)
    vol = v.astype(float)
    if manifold:
        vol = ndimage.gaussian_filter(vol, sigma=0.5)
    return np.ascontiguousarray(vol, dtype=np.float32)


last_mc33_stats = None   # of the last marching_cubes() call: [ambiguous cubes, resolved row != classic row, tunnels, interior tests]


def resolve_cube(values, level: float = 0.0):
    """Resolved triangle row of one cube (8 corner values): (triangles (n,3) int8 of cube-edge ids, J bits, tunnel, row)."""
    v = np.ascontiguousarray(np.asarray(values, dtype=np.float64) - level)
    out = np.full(36, -1, dtype=np.int8)
    info = np.zeros(3, dtype=np.int32)
    n = _mc_lib().t3d_oracle_resolve_cube(v.ctypes.data, out.ctypes.data, info.ctypes.data)
    return out[:3 * n].reshape(-1, 3).copy(), int(info[0]), int(info[1]), int(info[2])


def marching_cubes(vol32: np.ndarray, level: float = 0.5, want_hist: bool = False, z_base: int = 0):
    """skimage.measure.marching_cubes(volume, level) restated (oracle/mc_ref.c).

    Returns (verts float32 (V,3) [z,y,x], faces int32 (F,3), n_ambiguous[, case histogram]).
    Raises ValueError / RuntimeError exactly where skimage does (level outside range / no surface).
    z_base (test aid, 0 = skimage): vol32 is a z-slab starting at plane z_base of a larger volume; vertex z coordinates
    are formed from the global plane index, as a run on the whole volume would.
    """
    vol32 = np.ascontiguousarray(vol32, dtype=np.float32)
    if vol32.ndim != 3:
        raise ValueError("Input volume should be a 3D numpy array.")
    if vol32.shape[0] < 2 or vol32.shape[1] < 2 or vol32.shape[2] < 2:
        raise ValueError("Input array must be at least 2x2x2.")
    if level < vol32.min() or level > vol32.max():
        raise ValueError("Surface level must be within volume data range.")
    lib = _mc_lib()
    nz, ny, nx = vol32.shape
    nv, nf, na = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
    hist = np.zeros(256, dtype=np.int64) if want_hist else None
    rc = lib.t3d_oracle_marching_cubes(vol32.ctypes.data, nz, ny, nx, float(level), None, 0, None, 0,
                                       ctypes.byref(nv), ctypes.byref(nf), ctypes.byref(na),
                                       hist.ctypes.data if want_hist else None, None, int(z_base))
    if rc:
        raise RuntimeError("oracle marching cubes failed (%d)" % rc)
    if nf.value == 0:
        raise RuntimeError("No surface found at the given iso value.")
    verts = np.empty((nv.value, 3), dtype=np.float32)
    faces = np.empty((nf.value, 3), dtype=np.int32)
    stats = np.zeros(4, dtype=np.int64)
    rc = lib.t3d_oracle_marching_cubes(vol32.ctypes.data, nz, ny, nx, float(level),
                                       verts.ctypes.data, nv.value, faces.ctypes.data, nf.value,
                                       ctypes.byref(nv), ctypes.byref(nf), ctypes.byref(na), None, stats.ctypes.data, int(z_base))
    if rc:
        raise RuntimeError("oracle marching cubes failed (%d)" % rc)
    global last_mc33_stats
    last_mc33_stats = stats.tolist()
    if want_hist:
        return verts, faces, na.value, hist
    return verts, faces, na.value


def cube_cases(vol32: np.ndarray, level: float = 0.5) -> np.ndarray:
    vol32 = np.ascontiguousarray(vol32, dtype=np.float32)
    nz, ny, nx = vol32.shape
    out = np.empty((nz - 1, ny - 1, nx - 1), dtype=np.uint8)
    _mc_lib().t3d_oracle_cube_cases(vol32.ctypes.data, nz, ny, nx, float(level), out.ctypes.data)
    return out


def apply_variable_slice_depths(vertices: np.ndarray, slice_depths: np.ndarray, add_padding: bool = True) -> None:
    """surface_extractor.py:82-113, vectorised closed form (SURVEY.md V8, bit-exact vs the loop). In place."""
    if len(slice_depths) == 0:
        return
    slice_depths = np.asarray(slice_depths, dtype=np.float64)
    if add_padding:
        adj = np.concatenate([[slice_depths[0]], slice_depths, [slice_depths[-1]]])
    else:
        adj = slice_depths
    cum = np.cumsum(np.concatenate([[0], adj]))
    z = vertices[:, 0]
    lo = np.floor(z)
    neg = z < 0
    big = z >= len(cum) - 1
    mid = ~(neg | big)
    loi = lo[mid].astype(np.int64)
    frac = (z[mid] - lo[mid]).astype(np.float32)
    out = np.empty_like(z)
    out[neg] = 0
    out[big] = cum[-1]
    out[mid] = (cum[loi] + frac.astype(np.float64) * adj[np.minimum(loi, len(adj) - 1)]).astype(np.float32)
    vertices[:, 0] = out


def ensure_manifold_mesh(vertices: np.ndarray, faces: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """surface_extractor.py:115-126 (np.unique rows + drop faces with a repeated index)."""
    uv, inv = np.unique(vertices, axis=0, return_inverse=True)
    inv = np.asarray(inv).reshape(-1)
    nf = inv[faces]
    keep = (nf[:, 0] != nf[:, 1]) & (nf[:, 1] != nf[:, 2]) & (nf[:, 0] != nf[:, 2])
    return uv, nf[keep]


def extract_manifold_surface(volume_data, slice_depths, mm_per_pixel_y, mm_per_pixel_x,
                             smooth=True, manifold=True, add_padding=True,
                             return_diag: bool = False) -> Optional[Tuple[np.ndarray, np.ndarray]]:
    """surface_extractor.py:34-75 with skimage present."""
    try:
        vol32 = scalar_field(volume_data, manifold, add_padding)
        vertices, faces, n_amb = marching_cubes(vol32, 0.5)
        if manifold:
            vertices[:, 0] -= 1
            vertices[:, 1] -= 1
            vertices[:, 2] -= 1
        apply_variable_slice_depths(vertices, slice_depths, add_padding)
        vertices[:, 1] *= mm_per_pixel_y
        vertices[:, 2] *= mm_per_pixel_x
        if manifold:
            vertices, faces = ensure_manifold_mesh(vertices, faces)
        if return_diag:
            return vertices, faces, n_amb
        return vertices, faces
    except Exception:
        return None


def calculate_mesh_volume_f64(vertices: np.ndarray, faces: np.ndarray) -> float:
    """surface_extractor.py:128-139 evaluated in float64 (the parity definition, SURVEY.md fact 5)."""
    v = np.asarray(vertices, dtype=np.float64)
    a, b, c = v[faces[:, 0]], v[faces[:, 1]], v[faces[:, 2]]
    return float(abs(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6.0))


def calculate_mesh_volume_literal(vertices: np.ndarray, faces: np.ndarray):
    """surface_extractor.py:128-139 verbatim semantics (sequential; float32 accumulation under NumPy 2)."""
    volume = 0.0
    for face in faces:
        v0, v1, v2 = vertices[face[0]], vertices[face[1]], vertices[face[2]]
        volume += np.dot(v0, np.cross(v1, v2)) / 6.0
    return abs(volume)


def calculate_surface_area(vertices: np.ndarray, faces: np.ndarray):
    """surface_extractor.py:141-148."""
    v0, v1, v2 = vertices[faces[:, 0]], vertices[faces[:, 1]], vertices[faces[:, 2]]
    return np.sum(0.5 * np.linalg.norm(np.cross(v1 - v0, v2 - v0), axis=1))


def calculate_surface_area_f64(vertices: np.ndarray, faces: np.ndarray) -> float:
    v = np.asarray(vertices, dtype=np.float64)
    v0, v1, v2 = v[faces[:, 0]], v[faces[:, 1]], v[faces[:, 2]]
    return float(np.sum(0.5 * np.linalg.norm(np.cross(v1 - v0, v2 - v0), axis=1)))


# --------------------------------------------------------------------------------------------
# volume_calculator.py
# --------------------------------------------------------------------------------------------
def calculate_voxel_volume(voxel_data, mm_per_pixel_x, mm_per_pixel_y, mm_per_slice):
    """volume_calculator.py:16-21."""
    return np.sum(voxel_data) * (mm_per_pixel_x * mm_per_pixel_y * mm_per_slice)


def calculate_voxel_volume_variable_depth(voxel_data, mm_per_pixel_x, mm_per_pixel_y, slice_depths):
    """volume_calculator.py:23-35."""
    if len(slice_depths) == 0:
        return 0.0
    total = 0.0
    for z in range(min(voxel_data.shape[0], len(slice_depths))):
        total += np.sum(voxel_data[z]) * (mm_per_pixel_x * mm_per_pixel_y * slice_depths[z])
    return total


def calculate_bounding_box(voxel_data, mm_per_pixel_x, mm_per_pixel_y, mm_per_slice):
    """volume_calculator.py:37-57."""
    z, y, x = np.where(voxel_data)
    bx = (x.min() * mm_per_pixel_x, x.max() * mm_per_pixel_x)
    by = (y.min() * mm_per_pixel_y, y.max() * mm_per_pixel_y)
    bz = (z.min() * mm_per_slice, z.max() * mm_per_slice)
    return {"x": bx, "y": by, "z": bz, "dimensions": (bx[1] - bx[0], by[1] - by[0], bz[1] - bz[0])}


def calculate_bounding_box_variable_depth(voxel_data, mm_per_pixel_x, mm_per_pixel_y, slice_depths):
    """volume_calculator.py:59-94."""
    z, y, x = np.where(voxel_data)
    if len(z) == 0 or len(slice_depths) == 0:
        return {"x": (0, 0), "y": (0, 0), "z": (0, 0), "dimensions": (0, 0, 0)}
    bx = (x.min() * mm_per_pixel_x, x.max() * mm_per_pixel_x)
    by = (y.min() * mm_per_pixel_y, y.max() * mm_per_pixel_y)
    cum = np.cumsum(np.concatenate([[0], slice_depths]))
    bz = (cum[z.min()], cum[min(z.max() + 1, len(cum) - 1)])
    return {"x": bx, "y": by, "z": bz, "dimensions": (bx[1] - bx[0], by[1] - by[0], bz[1] - bz[0])}


# --------------------------------------------------------------------------------------------
# additive stage (no reference counterpart): exact Euclidean distance transform / SDF
# --------------------------------------------------------------------------------------------
def signed_distance(voxel_data: np.ndarray, sampling=(1.0, 1.0, 1.0)) -> np.ndarray:
    """sdf = edt(occ) - edt(~occ) (positive inside), voxel-centre distances, float32 (SURVEY.md a-16)."""
    occ = np.asarray(voxel_data, dtype=bool)
    if occ.all():
        inside = np.full(occ.shape, np.inf)
    else:
        inside = ndimage.distance_transform_edt(occ, sampling=sampling)
    if not occ.any():
        outside = np.full(occ.shape, np.inf)
    else:
        outside = ndimage.distance_transform_edt(~occ, sampling=sampling)
    return (inside - outside).astype(np.float32)


def squared_edt_index(voxel_data: np.ndarray) -> np.ndarray:
    """Exact integer squared distance (index space) from every set voxel to the nearest unset voxel."""
    occ = np.asarray(voxel_data, dtype=bool)
    d = ndimage.distance_transform_edt(occ)
    return np.rint(d * d).astype(np.int64)


# --------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md section 8d) -- shared by tests and bench
# --------------------------------------------------------------------------------------------
def ellipsoid_phantom_u8(Z: int, H: int, W: int, z0: int = 0, z1: Optional[int] = None) -> np.ndarray:
    """uint8 0/255 slices [z0, z1) of the analytic ellipsoid of SURVEY.md section 8d."""
    if z1 is None:
        z1 = Z
    cz, cy, cx = Z / 2 - 0.3, H / 2 + 0.2, W / 2 - 0.1
    rz, ry, rx = 0.42 * Z, 0.33 * H, 0.45 * W
    z = (np.arange(z0, z1, dtype=np.float64) - cz) / rz
    y = (np.arange(H, dtype=np.float64) - cy) / ry
    x = (np.arange(W, dtype=np.float64) - cx) / rx
    r2 = (z * z)[:, None, None] + (y * y)[None, :, None] + (x * x)[None, None, :]
    return np.where(r2 <= 1.0, np.uint8(255), np.uint8(0))


def reference_pipeline(masks_u8: np.ndarray, threshold: int, side_counts, total_depth_mm: float,
                       x_length_mm: float, y_length_mm: float, iterations: int = 3,
                       close_ends: bool = True, add_padding: bool = True) -> dict:
    """The whole hot path in the order tomography_3d_reconstruction.py runs it, once."""
    Z, H, W = masks_u8.shape
    masks = [masks_u8[z] >= threshold for z in range(Z)]  # image_loader.py:108
    vol = create_voxel_data(masks, close_ends)
    depths = calculate_slice_depths(total_depth_mm, *side_counts)
    mm_x, mm_y = x_length_mm / W, y_length_mm / H
    voxel_volume = calculate_voxel_volume_variable_depth(vol, mm_x, mm_y, depths)
    smoothed = smooth_voxel_data(vol, iterations, True)
    processed_volume = calculate_voxel_volume_variable_depth(smoothed, mm_x, mm_y, depths)
    res = extract_manifold_surface(smoothed, depths, mm_y, mm_x, True, True, add_padding, return_diag=True)
    out = {"voxel_data": vol, "smoothed": smoothed, "slice_depths": depths,
           "voxel_volume": voxel_volume, "processed_volume": processed_volume,
           "bbox": calculate_bounding_box_variable_depth(vol, mm_x, mm_y, depths)}
    if res is not None:
        v, f, namb = res
        out.update(vertices=v, faces=f, n_ambiguous=namb,
                   mesh_volume=calculate_mesh_volume_f64(v, f), surface_area=calculate_surface_area_f64(v, f))
    return out
