"""Pin the oracle against outputs of the UNMODIFIED reference modules (voxel_processor.py, surface_extractor.py,
volume_calculator.py) on seeded random inputs, for everything those modules compute without scikit-image.

tests/golden/reference_checks.npz holds the inputs and the expected outputs.  The outputs were recorded from the oracle:
this module used to import the reference from a separate checkout and assert the oracle's outputs on these same inputs
bit for bit equal to the reference's, and the oracle functions involved have not changed since.  Point clouds are
stored for subsample factor 1 only (a subsampled cloud is every k-th point of it); integer-valued arrays are stored in
the smallest integer type that holds them exactly."""
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _bbox_row(bb):
    return np.array([*bb["x"], *bb["y"], *bb["z"], *bb["dimensions"]], dtype=np.float64)


def test_close_volume_ends_and_volumes(gold, oracle):
    g = gold
    shapes, sides = g["v_shape"], g["v_sides"]
    n_vox = np.prod(shapes, axis=1)
    vols = np.unpackbits(g["v_vol"])[:n_vox.sum()].astype(bool)
    closed = np.unpackbits(g["v_closed"])[:n_vox.sum()].astype(bool)
    o_vox = np.concatenate([[0], np.cumsum(n_vox)])
    o_z = np.concatenate([[0], np.cumsum(shapes[:, 0])])
    o_pc = 0
    assert len(shapes) == 60
    for k, shape in enumerate(shapes):
        shape = tuple(int(s) for s in shape)
        vol = vols[o_vox[k]:o_vox[k + 1]].reshape(shape)
        expect = closed[o_vox[k]:o_vox[k + 1]].reshape(shape)
        d = g["v_depths"][o_z[k]:o_z[k + 1]]
        masks = [vol[z] for z in range(shape[0])]
        got = oracle.create_voxel_data(masks, True)
        assert np.array_equal(got, expect)
        assert np.array_equal(oracle.close_volume_ends_stencil(vol), expect)
        assert np.array_equal(oracle.calculate_slice_depths(6.0, *(int(s) for s in sides[k])), d)
        assert oracle.calculate_voxel_volume_variable_depth(expect, 0.3, 0.2, d) == g["v_volume"][k]
        assert np.array_equal(_bbox_row(oracle.calculate_bounding_box_variable_depth(expect, 0.3, 0.2, d)), g["v_bbox_var"][k])
        if expect.any():
            assert np.array_equal(_bbox_row(oracle.calculate_bounding_box(expect, 0.3, 0.2, 0.1)), g["v_bbox"][k])
        n_pc = int(expect.sum())
        pc = g["v_point_cloud"][o_pc:o_pc + n_pc]
        o_pc += n_pc
        for sub in (1, 2, 5):
            assert np.array_equal(oracle.generate_point_cloud(expect, 0.3, 0.2, d, sub), pc[::sub])
    assert o_pc == len(g["v_point_cloud"])


def test_surface_postprocessing(gold, oracle):
    g = gold
    depths = g["s_depths"]
    for pad in (True, False):
        key = "pad" if pad else "nopad"
        b = np.zeros((len(g["s_z_in_" + key]), 3), np.float32)
        b[:, 0] = g["s_z_in_" + key]
        oracle.apply_variable_slice_depths(b, depths, pad)
        assert np.array_equal(b[:, 0], g["s_z_out_" + key]) and not b[:, 1:].any()
    # vertices on a 0.37 grid (float32, many exact duplicates), random faces (some with repeated indices)
    verts = (g["s_grid"].astype(np.int64) * np.float32(0.37)).astype(np.float32)
    faces = g["s_faces"].astype(np.int32)
    ov, of = oracle.ensure_manifold_mesh(verts, faces)
    assert np.array_equal(ov, (g["s_manifold_grid"].astype(np.int64) * np.float32(0.37)).astype(np.float32))
    assert np.array_equal(of, g["s_manifold_faces"]) and of.dtype == np.int64
    small_f = of[:300]
    assert oracle.calculate_mesh_volume_literal(ov, small_f) == g["s_volume_literal"]
    assert oracle.calculate_surface_area(ov, of) == g["s_area"]
