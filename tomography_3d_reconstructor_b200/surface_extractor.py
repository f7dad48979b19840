#!/usr/bin/env python3
"""Drop-in `surface_extractor` module: the reference's SurfaceExtractor (surface_extractor.py:28-148) on sm_100a
kernels.  Same class / method names, parameter names/order and defaults, same prints, `None` on any extraction
failure (surface_extractor.py:74-75) -- except that a missing libt3d.so / CUDA device raises (no CPU fallback).

Returned vertices are float32 (V,3) [z_mm, y_mm, x_mm], lexicographically sorted and de-duplicated exactly like
np.unique(axis=0); faces are int64 (F,3) in the reference's cube order with degenerate faces dropped.  Both arrays
are READ-ONLY (copy them to edit): the device mesh they came from is recognised by array identity, so
calculate_mesh_volume / calculate_surface_area / the exporters do not upload them again.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import numpy as np

from . import engine


class SurfaceExtractor:
    """Handles surface extraction using marching cubes (B200)."""

    def __init__(self):
        self.last_error = None        # exception swallowed by the last extract_manifold_surface call, if any
        self.last_n_ambiguous = 0     # cubes whose tiling Lewiner's extra tests could have changed
        self.last_mesh = None         # engine.DeviceMesh of the last successful extraction

    def extract_manifold_surface(self, volume_data: np.ndarray, slice_depths: np.ndarray,
                                 mm_per_pixel_y: float, mm_per_pixel_x: float,
                                 smooth: bool = True, manifold: bool = True,
                                 add_padding: bool = True) -> Optional[Tuple[np.ndarray, np.ndarray]]:
        """Extract surface using marching cubes (surface_extractor.py:34-75).  `smooth` is unused, as in the reference."""
        self.last_error = None
        try:
            vertices, faces, _mesh = self._extract(volume_data, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold, add_padding, False)
            return vertices, faces

        except engine.T3DUnavailable:
            raise
        except Exception as e:  # reference behaviour: any failure -> None
            self.last_error = e
            if os.environ.get("T3D_RAISE"):
                raise
            return None

    def _extract(self, volume_data, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold, add_padding, normals):
        dv = engine.volume_from_host(volume_data)
        # the orchestrator extracts the same surface four times (tomography_3d_reconstruction.py:131,153,177,213,243):
        # memoise on the device volume (only volumes published by this package, which are read-only, can hit)
        sd = np.asarray(slice_depths, dtype=np.float64)
        key = ("extract", sd.tobytes(), repr(mm_per_pixel_y), repr(mm_per_pixel_x), type(mm_per_pixel_y).__name__,
               type(mm_per_pixel_x).__name__, bool(manifold), bool(add_padding))
        if normals:
            key += ("normals",)       # a mesh that keeps what its normals kernel reads
        cacheable = engine.volumes.lookup(volume_data) is dv
        mesh = dv.memo.get(key) if cacheable else None
        if mesh is None:
            mesh = engine.extract_surface(dv, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold, add_padding, normals=normals)
            if cacheable:
                dv.memo[key] = mesh
        vertices = engine.download(mesh.verts)      # fresh host arrays on every call, read-only: the device copy
        faces = engine.download(mesh.faces)         # is recognised by array identity (volume / area / export)
        vertices = engine.publish(engine.meshes, vertices, mesh)
        faces = engine.publish(engine.meshes, faces, mesh)
        self.last_mesh = mesh
        self.last_n_ambiguous = mesh.n_ambiguous

        print(f"Surface: {len(vertices)} vertices, {len(faces)} faces")

        return vertices, faces, mesh

    def extract_manifold_surface_ex(self, volume_data: np.ndarray, slice_depths: np.ndarray,
                                    mm_per_pixel_y: float, mm_per_pixel_x: float,
                                    smooth: bool = True, manifold: bool = True,
                                    add_padding: bool = True) -> Optional[Tuple[np.ndarray, np.ndarray, np.ndarray]]:
        """extract_manifold_surface plus the field-gradient vertex normals: (vertices, faces, normals), normals float32 (V,3)
        [z, y, x] unit vectors pointing out of the object, row i for vertex i (DESIGN.md §2).  Same prints, memo and `None`
        on failure; the three arrays are read-only."""
        self.last_error = None
        try:
            vertices, faces, mesh = self._extract(volume_data, slice_depths, mm_per_pixel_y, mm_per_pixel_x, manifold, add_padding, True)
            normals = engine.publish(engine.meshes, engine.download(mesh.normals), mesh)
            return vertices, faces, normals

        except engine.T3DUnavailable:
            raise
        except Exception as e:  # reference behaviour: any failure -> None
            self.last_error = e
            if os.environ.get("T3D_RAISE"):
                raise
            return None

    def calculate_mesh_volume(self, vertices: np.ndarray, faces: np.ndarray) -> float:
        """Calculate mesh volume using divergence theorem (surface_extractor.py:128-139); float64 accumulation."""
        if len(faces) == 0:
            return 0.0
        return abs(engine.mesh_from_host(vertices, faces).measures()[0])

    def calculate_surface_area(self, vertices: np.ndarray, faces: np.ndarray) -> float:
        """Calculate surface area from triangular faces (surface_extractor.py:141-148); float64 accumulation."""
        if len(faces) == 0:
            return 0.0
        return engine.mesh_from_host(vertices, faces).measures()[1]

    # ------------------------------------------------------------------------------------------------
    # additive API: the reference drops skimage's normals (surface_extractor.py:55 vs :72); they are exposed
    # here without widening the (vertices, faces) tuple
    def extract_surface_from_sdf(self, sdf, slice_depths: np.ndarray, mm_per_pixel_y: float, mm_per_pixel_x: float,
                                 level: float = 0.0, with_normals: bool = False):
        """Marching cubes on a signed distance field (positive inside, e.g. VoxelProcessor.compute_sdf) at `level`:
        vertices float32 [z_mm, y_mm, x_mm] (z through the variable slice depths, no padding), np.unique order, faces
        int64.  `sdf`: numpy float32 (Z,H,W) or a CUDA tensor.  with_normals=True: (vertices, faces, normals), the
        field-gradient unit normals of DESIGN.md §2 (pointing from field > level to field < level)."""
        import torch
        self.last_error = None
        try:
            f = sdf if isinstance(sdf, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(sdf, dtype=np.float32)).to(engine._require_cuda())
            mesh = engine.extract_surface(None, slice_depths, mm_per_pixel_y, mm_per_pixel_x, False, False, field=f.contiguous(),
                                          level=level, normals=with_normals)
            vertices, faces = engine.download(mesh.verts), engine.download(mesh.faces)
            vertices = engine.publish(engine.meshes, vertices, mesh)
            faces = engine.publish(engine.meshes, faces, mesh)
            self.last_mesh, self.last_n_ambiguous = mesh, mesh.n_ambiguous
            if with_normals:
                return vertices, faces, engine.publish(engine.meshes, engine.download(mesh.normals), mesh)
            return vertices, faces
        except engine.T3DUnavailable:
            raise
        except Exception as e:
            self.last_error = e
            if os.environ.get("T3D_RAISE"):
                raise
            return None

    def vertex_normals(self, vertices: np.ndarray, faces: np.ndarray) -> np.ndarray:
        """Area-weighted unit vertex normals, float32 (V,3) [z,y,x]."""
        from . import normals
        return normals.vertex_normals(engine.mesh_from_host(vertices, faces)).cpu().numpy()
