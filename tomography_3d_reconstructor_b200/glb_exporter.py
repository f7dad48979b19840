#!/usr/bin/env python3
"""Drop-in `glb_exporter` module: the reference's GLBExporter (glb_exporter.py:20-91).  `create_layer_colors` runs on the
device and `export_to_glb` writes the binary glTF file itself, from the device mesh (SURVEY.md 8f-3): no trimesh."""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import engine
from ._lib import check


class GLBExporter:
    """Handles exporting 3D models to GLB file format (B200)."""

    def __init__(self):
        pass

    def export_to_glb(self, vertices: np.ndarray, faces: np.ndarray, filename: str = "tomography_model.glb",
                      vertex_colors: Optional[np.ndarray] = None, vertex_normals: Optional[np.ndarray] = None) -> bool:
        """glb_exporter.py:26-50.  The reference hands the mesh to trimesh (Trimesh(...), fix_normals(), export 'glb');
        here the binary glTF 2.0 file is written directly: the binary chunk (uint32 indices, float32 positions, uint8
        RGBA COLOR_0) is assembled on the device from the mesh that is already there and downloaded once, the JSON
        chunk describes it.  Same prints and return values as the reference.  vertex_normals (float32 (V,3), e.g. from
        SurfaceExtractor.extract_manifold_surface_ex): written as the NORMAL attribute, for smooth shading."""
        try:
            write_glb(filename, vertices, faces, vertex_colors, vertex_normals)
            print(f"Model exported: {filename}")
            return True
        except engine.T3DUnavailable:
            raise
        except Exception as e:
            print(f"Export failed: {e}")
            return False

    def create_layer_colors(self, vertices: np.ndarray, slice_depths: np.ndarray, first_section1_slice: int,
                            last_section1_slice: int, highlight_thickness_mm: float = 1.0) -> np.ndarray:
        """Vertex colours (N,4) uint8 RGBA: grey, red within `highlight_thickness_mm` above the first Section_1 slice,
        blue above the last one (glb_exporter.py:52-91)."""
        n = len(vertices)
        if n == 0:
            return np.zeros((0, 4), dtype=np.uint8)
        cumulative_depths = np.cumsum(np.concatenate([[0], slice_depths]))
        has_a = first_section1_slice < len(cumulative_depths) - 1
        has_b = last_section1_slice < len(cumulative_depths) - 1
        a0 = float(cumulative_depths[first_section1_slice]) if has_a else 0.0
        b0 = float(cumulative_depths[last_section1_slice]) if has_b else 0.0
        a1 = float(cumulative_depths[first_section1_slice] + highlight_thickness_mm) if has_a else 0.0
        b1 = float(cumulative_depths[last_section1_slice] + highlight_thickness_mm) if has_b else 0.0
        mesh = engine.meshes.lookup(vertices)
        if mesh is not None and int(mesh.verts.shape[0]) == n:
            verts = mesh.verts.contiguous()
        else:
            verts = torch.from_numpy(np.ascontiguousarray(vertices, dtype=np.float32)).to(engine._require_cuda())
        out = torch.empty((n, 4), dtype=torch.uint8, device=verts.device)
        check(engine._L().t3d_layer_colors(engine._p(verts), n, 1 if has_a else 0, a0, a1, 1 if has_b else 0, b0, b1,
                                           engine._p(out), engine._stream()), "t3d_layer_colors")
        return engine.download(out)


def glb_bytes(vertices: np.ndarray, faces: np.ndarray, vertex_colors: Optional[np.ndarray] = None,
              vertex_normals: Optional[np.ndarray] = None) -> bytes:
    """The GLB file as bytes: 12-byte header, JSON chunk, BIN chunk (glTF 2.0 binary container).  vertex_normals: float32
    (V,3) [z,y,x] like the vertices, appended after the rest of the binary chunk as a NORMAL accessor; the normals point
    out of the object by definition, so the winding fix below leaves them as they are.  Without them the file is what it
    was before normals existed, byte for byte."""
    import json
    import struct
    L = engine._L()
    mesh = engine.mesh_from_host(vertices, faces)
    verts, fcs = mesh.verts.contiguous(), mesh.faces.contiguous()
    V, F = int(verts.shape[0]), int(fcs.shape[0])
    if V == 0 or F == 0:
        raise ValueError("empty mesh")
    dev = verts.device
    colors = None
    if vertex_colors is not None:
        c = np.ascontiguousarray(vertex_colors)
        if c.shape != (V, 4) or c.dtype != np.uint8:
            raise ValueError("vertex_colors must be (V, 4) uint8 RGBA")
        colors = torch.from_numpy(c).to(dev)
    normals = None
    if vertex_normals is not None:
        n = np.ascontiguousarray(vertex_normals)
        if n.shape != (V, 3) or n.dtype != np.float32:
            raise ValueError("vertex_normals must be (V, 3) float32")
        normals = torch.from_numpy(n).to(dev)
    # trimesh.fix_normals(): a closed, consistently wound mesh is turned inside out when its signed volume is negative
    signed_volume, _area = mesh.measures() if hasattr(mesh, "measures") else engine.mesh_measure(verts, fcs)
    flip = 1 if signed_volume < 0 else 0
    nbytes = int(L.t3d_glb_payload_bytes(V, F, 1 if colors is not None else 0))
    payload = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    minmax = torch.empty(6, dtype=torch.float32, device=dev)
    check(L.t3d_glb_pack(engine._p(verts), V, engine._p(fcs), F, 1 if fcs.dtype == torch.int64 else 0, engine._p(colors), flip,
                         engine._p(payload), engine._p(minmax), engine._stream()), "t3d_glb_pack")
    mm = minmax.cpu().tolist()
    if normals is not None:
        payload = torch.cat([payload, normals.view(-1).view(torch.uint8)])
    blob = engine.download(payload)
    views = [{"buffer": 0, "byteOffset": 0, "byteLength": 12 * F, "target": 34963},
             {"buffer": 0, "byteOffset": 12 * F, "byteLength": 12 * V, "target": 34962}]
    accessors = [{"bufferView": 0, "componentType": 5125, "count": 3 * F, "type": "SCALAR", "max": [V - 1], "min": [0]},
                 {"bufferView": 1, "componentType": 5126, "count": V, "type": "VEC3", "min": mm[:3], "max": mm[3:]}]
    attributes = {"POSITION": 1}
    if colors is not None:
        views.append({"buffer": 0, "byteOffset": 12 * F + 12 * V, "byteLength": 4 * V, "target": 34962})
        accessors.append({"bufferView": 2, "componentType": 5121, "normalized": True, "count": V, "type": "VEC4"})
        attributes["COLOR_0"] = 2
    if normals is not None:
        views.append({"buffer": 0, "byteOffset": nbytes, "byteLength": 12 * V, "target": 34962})
        accessors.append({"bufferView": len(views) - 1, "componentType": 5126, "count": V, "type": "VEC3"})
        attributes["NORMAL"] = len(accessors) - 1
        nbytes += 12 * V
    doc = {"asset": {"version": "2.0", "generator": "tomography_3d_reconstructor_b200"},
           "scene": 0, "scenes": [{"nodes": [0]}], "nodes": [{"name": "tomography_model", "mesh": 0}],
           "meshes": [{"name": "tomography_model", "primitives": [{"attributes": attributes, "indices": 0, "mode": 4}]}],
           "buffers": [{"byteLength": nbytes}], "bufferViews": views, "accessors": accessors}
    js = json.dumps(doc, separators=(",", ":")).encode("utf-8")
    js += b" " * (-len(js) % 4)
    pad = -nbytes % 4
    total = 12 + 8 + len(js) + 8 + nbytes + pad
    return b"".join([struct.pack("<4sII", b"glTF", 2, total), struct.pack("<I4s", len(js), b"JSON"), js,
                     struct.pack("<I4s", nbytes + pad, b"BIN\x00"), blob.tobytes(), b"\x00" * pad])


def write_glb(filename: str, vertices: np.ndarray, faces: np.ndarray, vertex_colors: Optional[np.ndarray] = None,
              vertex_normals: Optional[np.ndarray] = None) -> None:
    data = glb_bytes(vertices, faces, vertex_colors, vertex_normals)
    with open(filename, "wb") as f:
        f.write(data)


def parse_glb(data: bytes, with_normals: bool = False):
    """Minimal reader of what write_glb produces (used by the tests and tools/run_orchestrator.py to re-parse the file):
    returns (positions (V,3) f32, indices (F,3) u32, colours (V,4) u8 or None, json document); with_normals=True:
    (positions, indices, colours, normals (V,3) f32 or None, json document)."""
    import json
    import struct
    magic, version, total = struct.unpack_from("<4sII", data, 0)
    if magic != b"glTF" or version != 2 or total != len(data):
        raise ValueError("not a glTF 2.0 binary file")
    jlen, jtype = struct.unpack_from("<I4s", data, 12)
    doc = json.loads(data[20:20 + jlen].decode("utf-8"))
    blen, btype = struct.unpack_from("<I4s", data, 20 + jlen)
    if jtype != b"JSON" or btype != b"BIN\x00":
        raise ValueError("unexpected chunk types")
    blob = data[28 + jlen:28 + jlen + blen]
    prim = doc["meshes"][0]["primitives"][0]

    def read(acc_id, dtype, width):
        acc = doc["accessors"][acc_id]
        view = doc["bufferViews"][acc["bufferView"]]
        a = np.frombuffer(blob, dtype=dtype, count=acc["count"] * width, offset=view["byteOffset"])
        return a.reshape(-1, width) if width > 1 else a

    pos = read(prim["attributes"]["POSITION"], np.float32, 3)
    idx = read(prim["indices"], np.uint32, 1).reshape(-1, 3)
    col = read(prim["attributes"]["COLOR_0"], np.uint8, 4) if "COLOR_0" in prim["attributes"] else None
    if with_normals:
        nrm = read(prim["attributes"]["NORMAL"], np.float32, 3) if "NORMAL" in prim["attributes"] else None
        return pos, idx, col, nrm, doc
    return pos, idx, col, doc
