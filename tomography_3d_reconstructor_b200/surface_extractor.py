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

    def split_surface(self, vertices: np.ndarray, faces: np.ndarray) -> Tuple[np.ndarray, int]:
        """The connected bodies of a mesh, as scipy.sparse.csgraph.connected_components returns them for the graph with the
        edges f0-f1 and f0-f2 of every face: (int32 (V,) body of each vertex, number of bodies).  Bodies are numbered by their
        smallest vertex; a vertex no face uses is a body of its own."""
        bodies = engine.mesh_bodies(engine.mesh_from_host(vertices, faces))
        return engine.download(bodies.vertex_body()), bodies.n

    def analyze_surface_bodies(self, vertices: np.ndarray, faces: np.ndarray) -> dict:
        """Per-body arrays of a mesh (bodies as split_surface numbers them): n_bodies, vertex_counts, face_counts, first_vertex
        (int64), signed_volume_mm3, volume_mm3 (its absolute value) and surface_area_mm2 (float64, each an exactly summed
        divergence-theorem / area sum rounded once, DESIGN.md §2), bbox_mm (float32 (n, 6) [zmin, zmax, ymin, ymax, xmin,
        xmax]).  A hollow object gives two bodies whose signed volumes have opposite signs."""
        b = engine.mesh_bodies(engine.mesh_from_host(vertices, faces))
        sv = b.signed_volumes()
        return {"n_bodies": b.n, "vertex_counts": b.vertex_counts(), "face_counts": b.face_counts(), "first_vertex": b.first_vertex(),
                "signed_volume_mm3": sv, "volume_mm3": np.abs(sv), "surface_area_mm2": b.areas(), "bbox_mm": b.bbox_mm()}

    def filter_surface_bodies(self, vertices: np.ndarray, faces: np.ndarray, min_faces: int = 1, max_bodies=None,
                              vertex_normals: Optional[np.ndarray] = None):
        """The mesh of the bodies with at least min_faces faces; with max_bodies, only that many of the largest by face count
        (ties: the body with the smaller first vertex).  Vertices and faces keep their order and the faces their dtype, renumbered
        to the kept vertices.  Returns (vertices, faces), or (vertices, faces, normals) with the rows of vertex_normals that go
        with the kept vertices.  The arrays are read-only and, like extract_manifold_surface's, recognised by volume, area and
        the exporters without another upload."""
        mesh = engine.mesh_from_host(vertices, faces)
        bodies = engine.mesh_bodies(mesh)
        keep = engine.component_keep(bodies.face_counts(), min_faces, max_bodies) - 1
        normals = None
        if vertex_normals is not None:
            if engine.meshes.lookup(vertex_normals) is mesh and mesh.normals is not None:
                normals = mesh.normals
            else:
                import torch
                normals = torch.from_numpy(np.ascontiguousarray(vertex_normals, dtype=np.float32)).to(mesh.verts.device)
        out = bodies.select(keep, normals)
        v = engine.publish(engine.meshes, engine.download(out.verts), out)
        f = engine.publish(engine.meshes, engine.download(out.faces), out)
        if normals is None:
            return v, f
        return v, f, engine.publish(engine.meshes, engine.download(out.normals), out)

    def smooth_surface(self, vertices: np.ndarray, faces: np.ndarray, iterations: int = 10, lamb: float = 0.5, nu: float = 0.5
                       ) -> Tuple[np.ndarray, np.ndarray]:
        """Taubin smoothing of a mesh, as trimesh.smoothing.filter_taubin(mesh, lamb, nu, iterations) with its equal-weight
        Laplacian (bit for bit against the numpy definition of DESIGN.md §2), which takes the slice terraces and pixel
        staircase out of a marching-cubes surface while keeping its volume: (vertices float32 (V, 3), faces unchanged, in
        their dtype).  A vertex no face edge reaches keeps its position.  Both arrays are read-only and, like
        extract_manifold_surface's, recognised by volume, area, normals, bodies and the exporters without another upload;
        smoothing them again reuses the adjacency.  Raises ValueError for iterations < 0, a non-finite lamb or nu, or a face
        index outside [0, V)."""
        out = engine.smooth_mesh(engine.mesh_from_host(vertices, faces), iterations, lamb, nu)
        v = engine.publish(engine.meshes, engine.download(out.verts), out)
        f = engine.publish(engine.meshes, engine.download(out.faces), out)
        return v, f

    def vertex_normals(self, vertices: np.ndarray, faces: np.ndarray) -> np.ndarray:
        """Area-weighted unit vertex normals, float32 (V,3) [z,y,x]."""
        from . import normals
        return normals.vertex_normals(engine.mesh_from_host(vertices, faces)).cpu().numpy()
