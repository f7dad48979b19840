"""Mesh bodies on the device (engine.mesh_bodies, csrc/t3d_label.cu) against tests/bodies_oracle.py, bit for bit: labels,
body count, counts, first vertex, boxes, exactly summed signed volumes and areas, face bodies and selected meshes, on meshes
from every extraction path and from the host; the body filter of SurfaceExtractor through the identity registry and the
exporters; the refusals."""
import numpy as np
import pytest

import bodies_oracle as bo
from conftest import random_blobs

gpu = pytest.mark.gpu

MM_Y, MM_X = 0.29, 0.37


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def check_bodies(eng, mesh, n_min=1, n_max=None):
    """mesh_bodies(mesh) against the oracle, and select() of every other body and of the largest; returns (bodies, oracle)."""
    v, f = mesh.verts.cpu().numpy(), mesh.faces.cpu().numpy()
    b = eng.mesh_bodies(mesh)
    lab, n = bo.labels(f, len(v))
    assert b.n == n and n_min <= n and (n_max is None or n <= n_max)
    assert bits_equal(b.vertex_body().cpu().numpy(), lab)
    want = bo.stats(v, f, lab, n)
    for name in ("vertex_counts", "face_counts", "first_vertex", "bbox_mm", "signed_volumes", "areas"):
        assert bits_equal(getattr(b, name)(), want[name]), name
    assert bits_equal(b.face_body().cpu().numpy(), want["face_body"])
    largest = [int(np.argmax(want["face_counts"]))] if n else []
    for keep in (list(range(0, n, 2)), largest, []):
        out = b.select(keep)
        sv, sf = bo.select(v, f, lab, keep)
        assert bits_equal(out.verts.cpu().numpy(), sv) and bits_equal(out.faces.cpu().numpy(), sf), keep[:5]
    return b, want


def extracted(vol, manifold=True, add_padding=True, depths=None):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor, engine
    se = SurfaceExtractor()
    d = np.linspace(0.4, 0.9, vol.shape[0]) if depths is None else depths
    v, f = se.extract_manifold_surface(vol, d, MM_Y, MM_X, True, manifold, add_padding)
    return engine.mesh_from_host(v, f), se


def ellipsoid(shape, centre, radii):
    z, y, x = np.indices(shape, dtype=np.float64)
    return sum(((c - m) / r) ** 2 for c, m, r in zip((z, y, x), centre, radii)) <= 1.0


@gpu
def test_phantom_is_one_body_with_the_whole_mesh_measures(eng, oracle):
    vol = oracle.smooth_voxel_data(oracle.ellipsoid_phantom_u8(24, 64, 96) >= 200, 3, True)
    mesh, _ = extracted(vol)
    b, want = check_bodies(eng, mesh, 1, 1)
    sv, sa = mesh.measures()
    assert abs(b.signed_volumes()[0] - sv) <= 1e-12 * abs(sv) and abs(b.areas()[0] - sa) <= 1e-12 * sa
    assert b.first_vertex()[0] == 0 and b.vertex_counts()[0] == len(mesh.verts)


@gpu
def test_two_ellipsoids_and_a_hollow_one(eng):
    shape = (30, 60, 90)
    two = ellipsoid(shape, (15, 30, 22), (10, 20, 15)) | ellipsoid(shape, (15, 30, 68), (8, 18, 14))
    b, want = check_bodies(eng, extracted(two)[0], 2, 2)
    assert (b.signed_volumes() > 0).all() or (b.signed_volumes() < 0).all()
    hollow = ellipsoid(shape, (15, 30, 45), (12, 25, 38)) & ~ellipsoid(shape, (15, 30, 45), (6, 12, 20))
    mesh, _ = extracted(hollow)
    b, want = check_bodies(eng, mesh, 2, 2)
    s = b.signed_volumes()
    assert s[0] * s[1] < 0                                    # outer shell and cavity shell have opposite signs
    assert b.bbox_mm()[0, 5] > b.bbox_mm()[1, 5]              # body 0 (the smallest vertex) is the outer shell
    sv, _ = mesh.measures()
    assert abs((s[0] + s[1]) - sv) <= 1e-9 * abs(sv)          # the cavity subtracts from the whole-mesh volume


@gpu
def test_blobs_noise_and_open_bodies(eng):
    rng = np.random.default_rng(31)
    check_bodies(eng, extracted(random_blobs(rng, (28, 64, 96), 0.12, 2.0))[0], 6)
    noise = rng.random((40, 96, 128)) < 0.2                 # unsmoothed: isolated voxels, ambiguous cubes
    mesh, se = extracted(noise)
    assert se.last_n_ambiguous > 0
    check_bodies(eng, mesh, 1000)
    touching = random_blobs(rng, (20, 48, 70), 0.4, 1.5)    # objects cut by the volume's faces: open bodies
    touching[:, :, 0] = True
    check_bodies(eng, extracted(touching, add_padding=False)[0], 1)


@gpu
def test_raw_int32_and_sdf_meshes(eng, oracle):
    import torch
    from tomography_3d_reconstructor_b200 import SurfaceExtractor, VoxelProcessor
    rng = np.random.default_rng(37)
    vol = random_blobs(rng, (22, 50, 80), 0.25, 1.5)
    dv = eng.volume_from_host(vol)
    raw = eng.extract_surface(dv, np.linspace(0.5, 1.0, 22), MM_Y, MM_X, manifold=False)
    assert raw.faces.dtype == torch.int32
    check_bodies(eng, raw, 2)
    sdf = VoxelProcessor().compute_sdf(vol, (0.7, MM_Y, MM_X))
    se = SurfaceExtractor()
    v, f = se.extract_surface_from_sdf(sdf, np.full(22, 0.7), MM_Y, MM_X, 0.0)
    check_bodies(eng, eng.mesh_from_host(v, f), 2)


def host_mesh(rng, V, F, clusters):
    cl = rng.integers(0, clusters, V)
    faces = []
    for c in range(clusters):
        m = np.flatnonzero(cl == c)
        if len(m):
            faces.append(rng.choice(m, (F // clusters, 3)))
    f = np.concatenate(faces) if faces else np.zeros((0, 3), np.int64)
    keep_out = rng.random(V) < 0.1                           # unreferenced vertices
    f = f[~keep_out[f].any(axis=1)]
    v = (rng.standard_normal((V, 3)) * 50).astype(np.float32)
    v[rng.random((V, 3)) < 0.02] = -0.0
    return v, f


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_host_meshes_random_connectivity_and_empty(eng, dtype):
    import torch
    rng = np.random.default_rng(41)
    for V, F, k in ((5000, 6000, 40), (70000, 200000, 3), (300, 50, 300), (1, 1, 1)):
        v, f = host_mesh(rng, V, F, k)
        check_bodies(eng, eng.mesh_from_host(v, f.astype(dtype)))
    dev = torch.device("cuda")
    empty = eng.DeviceMesh(torch.zeros((0, 3), dtype=torch.float32, device=dev), torch.zeros((0, 3), dtype=torch.int64, device=dev))
    b = check_bodies(eng, empty, 0, 0)[0]
    assert b.n == 0 and b.select([]).verts.shape[0] == 0
    lone = eng.mesh_from_host(np.ones((4, 3), np.float32), np.zeros((0, 3), dtype))
    b = check_bodies(eng, lone, 4, 4)[0]
    assert b.face_counts().tolist() == [0] * 4 and b.first_vertex().tolist() == [0, 1, 2, 3]


@gpu
def test_repeated_and_fresh_copies_are_identical(eng):
    rng = np.random.default_rng(43)
    mesh, _ = extracted(rng.random((30, 80, 100)) < 0.25)
    b1 = eng.mesh_bodies(mesh)
    assert eng.mesh_bodies(mesh) is b1
    fresh = eng.DeviceMesh(mesh.verts.clone(), mesh.faces.clone())
    b2 = eng.mesh_bodies(fresh)
    assert b2 is not b1 and b2.n == b1.n
    assert bits_equal(b1.vertex_body().cpu().numpy(), b2.vertex_body().cpu().numpy())
    for name in ("vertex_counts", "face_counts", "first_vertex", "bbox_mm", "signed_volumes", "areas"):
        assert bits_equal(getattr(b1, name)(), getattr(b2, name)()), name


@gpu
def test_filter_keeps_the_phantom_without_its_debris(eng, oracle, tmp_path):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    from tomography_3d_reconstructor_b200.glb_exporter import glb_bytes, parse_glb
    from tomography_3d_reconstructor_b200.obj_exporter import OBJExporter
    phantom = oracle.smooth_voxel_data(oracle.ellipsoid_phantom_u8(24, 64, 96) >= 200, 3, True)    # one body
    debris = phantom.copy()
    debris[2:5, 1:4, 1:4] = True                              # cubes at least five voxels from the ellipsoid
    debris[18:21, 60:63, 91:94] = True
    debris[10:12, 1:3, 90:92] = True
    se = SurfaceExtractor()
    d = np.linspace(0.4, 0.9, 24)
    v, f, n = se.extract_manifold_surface_ex(debris, d, MM_Y, MM_X)
    pv, pf, pn = se.extract_manifold_surface_ex(phantom, d, MM_Y, MM_X)
    info = se.analyze_surface_bodies(v, f)
    assert info["n_bodies"] == 4 and info["face_counts"].max() == len(pf)
    assert np.array_equal(info["volume_mm3"], np.abs(info["signed_volume_mm3"]))
    v2, f2, n2 = se.filter_surface_bodies(v, f, max_bodies=1, vertex_normals=n)
    assert bits_equal(v2, pv) and bits_equal(f2, pf) and bits_equal(n2, pn)
    lab, _ = se.split_surface(v, f)
    assert bits_equal(lab, bo.labels(f, len(v))[0])
    assert bits_equal(n2, bo.select(v, f, lab, [int(np.argmax(info["face_counts"]))], n)[2])
    assert not v2.flags.writeable and eng.meshes.lookup(v2) is eng.meshes.lookup(f2) is not None
    assert se.calculate_mesh_volume(v2, f2) == se.calculate_mesh_volume(pv, pf)
    # host normals (not from the registry) are uploaded and go along the same way; without normals two arrays come back
    v3, f3, n3 = se.filter_surface_bodies(v, f, max_bodies=1, vertex_normals=np.array(n))
    assert bits_equal(n3, n2) and len(se.filter_surface_bodies(v, f, min_faces=10 ** 9)) == 2
    pos, idx, _col, nrm, _doc = parse_glb(glb_bytes(v2, f2, vertex_normals=n2), with_normals=True)
    assert bits_equal(pos, v2) and bits_equal(nrm, n2)
    assert np.array_equal(idx.astype(np.int64), f2) or np.array_equal(idx.astype(np.int64), f2[:, [0, 2, 1]])
    a, b = str(tmp_path / "a.obj"), str(tmp_path / "b.obj")
    assert OBJExporter().export_to_obj(v2, f2, a) and OBJExporter().export_to_obj(np.array(v2), np.array(f2), b)
    assert open(a, "rb").read() == open(b, "rb").read()


@gpu
def test_full_size_c1_phantom_mesh(eng):
    import torch
    from bench import PHYS, THRESHOLD, make_phantom_u8, side_counts
    from tomography_3d_reconstructor_b200 import pipeline
    Z, H, W = 512, 1024, 1024
    masks = make_phantom_u8(Z, H, W, 0, Z, torch.device("cuda"))
    out = pipeline.reconstruct_fused(masks, THRESHOLD, side_counts(Z), PHYS["total_depth_mm"], PHYS["x_length_mm"], PHYS["y_length_mm"])
    del masks
    mesh = out["mesh"]
    assert mesh.faces.shape[0] > 3_000_000
    b, _ = check_bodies(eng, mesh, 1, 1)
    sv, sa = mesh.measures()
    assert abs(b.signed_volumes()[0] - sv) <= 1e-12 * abs(sv) and abs(b.areas()[0] - sa) <= 1e-12 * sa


@gpu
def test_refusals(eng):
    from tomography_3d_reconstructor_b200._lib import T3DError
    v = np.array([[1e30, 0, 0], [0, 1e30, 0], [0, 0, 1e30]], np.float32)
    with pytest.raises(T3DError, match="2\\^62"):
        eng.mesh_bodies(eng.mesh_from_host(v, np.array([[0, 1, 2]])))
    with pytest.raises(ValueError):
        eng.mesh_bodies(eng.mesh_from_host(v, np.array([[0, 1, 3]])))


# ---- host only --------------------------------------------------------------------------------------------------------
def test_int32_limits_are_refused_with_the_count():
    """Beyond int32 vertices or faces the calls return status 2 naming the count, before they touch any memory."""
    import os
    from tomography_3d_reconstructor_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    lib = _lib.load()
    n = 2 ** 31 + 5
    assert lib.t3d_mesh_bodies_label(None, 0, 0, n, None, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
    assert lib.t3d_mesh_bodies_stats(None, None, n, 0, 10, None, 3, None, None, None, None, None, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
    assert lib.t3d_mesh_bodies_stats(None, None, 0, 0, 10, None, 11, None, None, None, None, None, None, None, None) == 2
    assert lib.t3d_mesh_bodies_select(None, None, None, 0, 0, n, None, 1, None, None, None, None, None, None) == 2
