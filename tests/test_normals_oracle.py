"""The normals oracle (tests/normals_oracle.py) rebuilds the vertices from the cut edges of the marched field on its own:
they must be exactly the vertices of oracle.extract_manifold_surface, and its tie rule must be exercised by a field whose
cut edges collapse onto one node."""
import numpy as np
import pytest

from conftest import random_blobs
import normals_oracle as no

MM = (0.19, 0.28)


def _phantom(Z, H, W):
    from oracle import cpu_ref
    return cpu_ref.smooth_voxel_data(cpu_ref.ellipsoid_phantom_u8(Z, H, W) >= 200, 3, True)


def _touching():
    """An object touching slice 0 and the x / y borders: the z-clamp group and the reflect boundary."""
    rng = np.random.default_rng(7)
    v = random_blobs(rng, (9, 21, 27), 0.45, 1.2)
    v[0, 3:15, 0:9] = True
    v[:4, 0:6, 20:27] = True
    return v


def volumes():
    from oracle import cpu_ref
    depths_c0 = np.array([0.009375] * 20 + [0.09375] * 64 + [0.009375] * 20)
    rng = np.random.default_rng(3)
    noise = random_blobs(rng, (11, 19, 23), 0.5, 0.6)
    return {
        "ellipsoid_20_64_20": (_phantom(104, 40, 48), depths_c0, True),
        "no_padding": (_phantom(24, 36, 44), cpu_ref.calculate_slice_depths(6.0, 3, 18, 3), False),
        "no_z_map": (_phantom(16, 30, 34), np.array([]), True),
        "noise_ambiguous": (noise, cpu_ref.calculate_slice_depths(4.0, 2, 7, 2), True),
        "touching_slice0_and_border": (_touching(), cpu_ref.calculate_slice_depths(3.0, 2, 5, 2), True),
    }


@pytest.mark.parametrize("name", list(volumes()))
def test_cut_edge_vertices_are_the_reference_vertices(oracle, name):
    vol, depths, add_padding = volumes()[name]
    ref = oracle.extract_manifold_surface(vol, depths, MM[0], MM[1], True, True, add_padding)
    assert ref is not None
    f = oracle.scalar_field(vol, True, add_padding)
    verts, lo, axes, t, fz = no.cut_edge_vertices(f, 0.5, depths, MM[0], MM[1], add_padding, unpad=True)
    uv = np.unique(verts, axis=0)
    assert uv.dtype == np.float32 and np.array_equal(uv.view(np.uint32), ref[0].view(np.uint32))
    v2, n2 = no.gradient_normals(vol, depths, MM[0], MM[1], True, add_padding)
    assert np.array_equal(v2.view(np.uint32), ref[0].view(np.uint32)) and n2.shape == v2.shape
    nn = np.linalg.norm(n2.astype(np.float64), axis=1)
    assert np.all(np.abs(nn - 1) < 1e-6)


def test_touching_case_has_a_clamp_group(oracle):
    vol, depths, add_padding = volumes()["touching_slice0_and_border"]
    f = oracle.scalar_field(vol, True, add_padding)
    verts, lo, axes, t, fz = no.cut_edge_vertices(f, 0.5, depths, MM[0], MM[1], add_padding, unpad=True)
    assert (fz < 0).any() and (verts[:, 0] == 0).sum() > (fz < 0).sum()


def tie_field():
    """Dense float32 field (level 0.5): a ball plus one isolated node one ulp above the level.  Its six cut edges all
    round onto the node, so np.unique merges six raw vertices whose normals point six different ways."""
    Z, H, W = 12, 12, 18
    z, y, x = np.meshgrid(np.arange(Z), np.arange(H), np.arange(W), indexing="ij")
    f = (0.5 + 3.2 - np.sqrt((z - 5.5) ** 2 + (y - 6.0) ** 2 + (x - 5.0) ** 2)).astype(np.float32)
    f[6, 6, 14] = np.nextafter(np.float32(0.5), np.float32(1))
    return f, 0.5


def test_tie_rule_runs_on_a_collapsing_node():
    f, level = tie_field()
    depths = np.linspace(0.5, 1.5, f.shape[0])
    verts, lo, axes, t, fz = no.cut_edge_vertices(f, level, depths, MM[0], MM[1], False, unpad=False)
    n = no.raw_normals(f, level, lo, axes, t, fz, depths, MM[0], MM[1], False)
    at_node = np.all(lo == [6, 6, 14], axis=1) | (np.all(lo == [5, 6, 14], axis=1) & (axes == 0)) | \
        (np.all(lo == [6, 5, 14], axis=1) & (axes == 1)) | (np.all(lo == [6, 6, 13], axis=1) & (axes == 2))
    assert at_node.sum() == 6
    node_verts = np.unique(verts[at_node], axis=0)
    assert len(node_verts) == 1                                  # all six round onto the node
    assert len(np.unique(n[at_node], axis=0)) == 6              # ... with six different normals
    uv, un, merged = no.gradient_normals_dense(f, level, depths, MM[0], MM[1])
    assert merged == 5
    slot = np.nonzero(np.all(uv == node_verts[0], axis=1))[0][0]
    keys = no.edge_keys(lo, axes)
    win = np.nonzero(at_node)[0][np.argmin(keys[at_node])]
    assert axes[win] == 0 and tuple(lo[win]) == (5, 6, 14)    # the z edge from below has the smallest key
    assert np.array_equal(un[slot], n[win])
