"""ctypes binding of libt3d.so (C ABI declared in include/t3d.h).

The library is built in-tree by __graft_entry__.build() (nvcc, sm_100a).  There is no CPU fallback: if the
shared object is missing or a CUDA device is not available the product path raises.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libt3d.so")

_c = ctypes
_vp, _i, _i64, _u32, _dbl = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_uint32, _c.c_double

class McField(ctypes.Structure):
    """struct t3d_mc_field (include/t3d.h): the marched field as the ambiguity tests of marching cubes see it."""
    _fields_ = [("occ_bits", _vp), ("Z", _i), ("H", _i), ("W", _i), ("pad", _i), ("gaussian", _i), ("weights3_host", _vp),
                ("field_f32", _vp), ("level", _dbl)]


# name -> (restype, argtypes); mirrors include/t3d.h one to one (tests/test_abi.py checks both directions)
SIGNATURES = {
    "t3d_last_error": (_c.c_char_p, []),
    "t3d_version": (_i, []),
    "t3d_words_per_row": (_i64, [_i]),
    "t3d_launch_count": (_i64, []),
    "t3d_count_launches": (None, [_i]),
    "t3d_pack_masks": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "t3d_pack_gap": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_unpack_bits": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "t3d_fill_holes_scratch_bytes": (_i64, [_i, _i, _i]),
    "t3d_fill_holes_2d": (_i, [_vp, _i, _i64, _i, _i, _vp, _vp]),
    "t3d_gap_fill": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "t3d_morph_scratch_bytes": (_i64, [_i, _i, _i, _i]),
    "t3d_morph": (_i, [_vp, _vp, _i, _i, _i, _i, _c.c_uint, _vp, _vp, _vp]),
    "t3d_volume_stats": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
    "t3d_row_popcounts": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "t3d_point_cloud_emit": (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _dbl, _dbl, _vp, _vp]),
    "t3d_scan_workspace_bytes": (_i64, [_i64, _i]),
    "t3d_field_sign": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_field_sign_lean": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _u32, _vp, _vp]),
    "t3d_mc_num_chunks": (_i64, [_i, _i, _i]),
    "t3d_mc_flags": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "t3d_field_dense": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "t3d_cube_cases": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "t3d_canonicalize_workspace_bytes": (_i64, [_i64, _i64]),
    "t3d_mesh_canonicalize": (_i, [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "t3d_canonicalize_fast_workspace_bytes": (_i64, [_i64, _i64]),
    "t3d_mesh_measure_workspace_bytes": (_i64, []),
    "t3d_exclusive_scan_u32_dev": (_i, [_vp, _vp, _i64, _i64, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_mc_words_dev": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "t3d_mc_emit_dev": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _u32, _vp, _u32, _u32, _vp, _vp, _i, _vp, _vp]),
    "t3d_mc_vertices_dev": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _dbl, _vp, _vp, _u32, _i, _i, _vp, _vp, _i, _dbl, _dbl, _i, _i, _vp,
                                 _vp]),
    "t3d_mesh_canonicalize_fast_dev": (_i, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "t3d_mesh_measure_dev": (_i, [_vp, _vp, _i64, _vp, _i, _vp, _vp, _vp]),
    "t3d_canonicalize_structured_workspace_bytes": (_i64, [_i64, _i64, _u32, _u32, _i]),
    "t3d_mesh_canonicalize_structured_dev": (_i, [_vp, _vp, _i64, _vp, _vp, _i, _i, _i, _vp, _vp, _u32, _i, _i, _vp, _vp, _i, _i, _u32,
                                                  _u32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    "t3d_reconstruct_workspace_bytes": (_i64, [_i, _i, _i, _i, _i, _u32, _u32, _u32, _u32, _u32]),
    "t3d_reconstruct_results_len": (_i64, [_i]),
    "t3d_reconstruct": (_i, [_vp, _i, _i, _i, _i, _i, _i, _c.c_uint, _i, _vp, _vp, _vp, _i, _dbl, _dbl, _i, _u32, _u32, _u32,
                             _u32, _u32, _i, _vp, _vp, _vp, _vp, _vp]),
    "t3d_reconstruct_slab_workspace_bytes": (_i64, [_i, _i, _i, _i, _i, _i, _i, _u32, _u32, _u32, _u32, _u32]),
    "t3d_slab_pack_gap_ok": (_i, [_vp, _i, _i, _i, _i]),
    "t3d_slab_pack": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "t3d_reconstruct_slab": (_i, [_vp, _i, _i, _i, _i, _i, _i, _c.c_uint, _i, _i, _i, _i, _i, _c.c_float, _i, _c.c_float, _i, _vp, _vp,
                                  _vp, _i, _dbl, _dbl, _i, _u32, _u32, _u32, _u32, _u32, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "t3d_slab_stitch_faces": (_i, [_vp, _i64, _vp, _i64, _i, _vp]),
    "t3d_edt_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_edt_xy_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_edt_xy": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_edt_z_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_edt_z": (_i, [_vp, _vp, _i, _i, _i, _vp, _c.c_float, _i, _vp, _vp, _vp]),
    "t3d_edt": (_i, [_vp, _i, _i, _i, _i, _vp, _c.c_float, _i, _vp, _vp, _vp]),
    "t3d_endcap_slices": (_i, [_vp, _i, _i, _vp, _i, _vp, _vp]),
    "t3d_sdf_xy_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_sdf_xy": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_sdf_z_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_sdf_z": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_sdf_workspace_bytes": (_i64, [_i, _i, _i]),
    "t3d_sdf": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "t3d_sign_from_f32": (_i, [_vp, _i, _i, _i, _dbl, _vp, _vp]),
    "t3d_layer_colors": (_i, [_vp, _i64, _i, _dbl, _dbl, _i, _dbl, _dbl, _vp, _vp]),
    "t3d_obj_workspace_bytes": (_i64, [_i64, _i64]),
    "t3d_glb_payload_bytes": (_i64, [_i64, _i64, _i]),
    "t3d_glb_pack": (_i, [_vp, _i64, _vp, _i64, _i, _vp, _i, _vp, _vp, _vp]),
    "t3d_obj_measure": (_i, [_vp, _i64, _vp, _i64, _i, _vp, _vp, _vp]),
    "t3d_obj_emit": (_i, [_vp, _i64, _vp, _i64, _i, _vp, _vp, _vp, _vp]),
    "t3d_vertex_normals": (_i, [_vp, _i64, _vp, _i64, _i, _vp, _vp]),
    "t3d_mc_normals_dev": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _dbl, _vp, _vp, _u32, _i, _i, _vp, _i, _dbl, _dbl, _vp, _vp,
                                _vp, _vp, _vp, _vp]),
    "t3d_canonical_map_offsets": (_i, [_i, _i64, _i64, _u32, _u32, _i, _vp]),
    "t3d_reconstruct_normals": (_i, [_i, _i, _i, _i, _c.c_uint, _i, _vp, _vp, _i, _dbl, _dbl, _u32, _u32, _u32, _u32, _u32, _vp, _vp,
                                     _vp, _vp]),
}


class T3DError(RuntimeError):
    pass


_lib = None


def load():
    """Load libt3d.so and attach the prototypes.  Raises (never falls back) if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise T3DError(
            "libt3d.so not found at %s -- run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().t3d_last_error()
        raise T3DError("%s failed (%d): %s" % (what or "libt3d call", rc, msg.decode() if msg else "?"))
