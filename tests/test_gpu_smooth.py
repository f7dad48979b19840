"""Mesh smoothing on the device (engine.vertex_neighbors / engine.smooth_mesh, csrc/t3d_smooth.cu) against
tests/smooth_oracle.py, bit for bit: CSR offsets, neighbours and smoothed vertices on meshes from every extraction path and
from the host, rows on both sides of the warp sort and far beyond it, empty meshes and the full C1 mesh; repeatability; the
smoothed surface of SurfaceExtractor through the identity registry, the measures, bodies and the exporters; the refusals."""
import numpy as np
import pytest

import bodies_oracle as bo
import smooth_oracle as so
from conftest import random_blobs

gpu = pytest.mark.gpu

MM_Y, MM_X = 0.29, 0.37
PARAMS = [(0, 0.5, 0.5), (1, 0.5, 0.5), (2, 0.5, 0.5), (10, 0.5, 0.5), (25, 0.5, 0.5), (6, 0.33, 0.34), (3, 0.6, -0.1)]


def bits_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def check_smooth(eng, mesh, params=((10, 0.5, 0.5),)):
    """vertex_neighbors(mesh) and smooth_mesh(mesh, *p) for every p against the oracle; returns the oracle's CSR arrays."""
    v, f = mesh.verts.cpu().numpy(), mesh.faces.cpu().numpy()
    off, nb = eng.vertex_neighbors(mesh)
    want_off, want_nb = so.adjacency(f, len(v))
    assert bits_equal(off.cpu().numpy(), want_off) and bits_equal(nb.cpu().numpy(), want_nb)
    for it, lamb, nu in params:
        out = eng.smooth_mesh(mesh, it, lamb, nu)
        assert out.faces is mesh.faces and out._adjacency is mesh._adjacency and out.normals is None
        assert bits_equal(out.verts.cpu().numpy(), so.taubin(v, want_off, want_nb, it, lamb, nu)), (it, lamb, nu)
    return want_off, want_nb


def extracted(vol, manifold=True, add_padding=True):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor, engine
    se = SurfaceExtractor()
    v, f = se.extract_manifold_surface(vol, np.linspace(0.4, 0.9, vol.shape[0]), MM_Y, MM_X, True, manifold, add_padding)
    return engine.mesh_from_host(v, f)


def ellipsoid(shape, centre, radii):
    z, y, x = np.indices(shape, dtype=np.float64)
    return sum(((c - m) / r) ** 2 for c, m, r in zip((z, y, x), centre, radii)) <= 1.0


def raw_row_lengths(faces, V):
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    e = e[e[:, 0] != e[:, 1]]
    return np.bincount(e.ravel(), minlength=V)


@pytest.fixture(scope="module")
def phantom(oracle):
    return oracle.smooth_voxel_data(oracle.ellipsoid_phantom_u8(24, 64, 96) >= 200, 3, True)


@gpu
def test_phantom_every_parameter_set(eng, phantom):
    mesh = extracted(phantom)
    check_smooth(eng, mesh, PARAMS)
    sv, sa = mesh.measures()
    out = eng.smooth_mesh(mesh)
    tv, ta = out.measures()
    assert ta < sa and abs(tv - sv) <= 1e-3 * abs(sv)


@gpu
def test_hollow_ellipsoid_and_open_mesh(eng):
    shape = (30, 60, 90)
    hollow = ellipsoid(shape, (15, 30, 45), (12, 25, 38)) & ~ellipsoid(shape, (15, 30, 45), (6, 12, 20))
    check_smooth(eng, extracted(hollow), PARAMS[1:4])
    touching = random_blobs(np.random.default_rng(53), (20, 48, 70), 0.4, 1.5)
    touching[:, :, 0] = True
    check_smooth(eng, extracted(touching, add_padding=False), PARAMS[2:4])


@gpu
@pytest.mark.parametrize("density", [0.1, 0.3, 0.5])
def test_unsmoothed_noise(eng, density):
    mesh = extracted(np.random.default_rng(59).random((24, 64, 64)) < density)
    if density == 0.5:
        assert raw_row_lengths(mesh.faces.cpu().numpy(), mesh.verts.shape[0]).max() > 32
    check_smooth(eng, mesh, PARAMS[3:4] + PARAMS[5:6])


@gpu
def test_raw_int32_and_sdf_meshes(eng):
    import torch
    from tomography_3d_reconstructor_b200 import SurfaceExtractor, VoxelProcessor
    vol = random_blobs(np.random.default_rng(61), (22, 50, 80), 0.25, 1.5)
    raw = eng.extract_surface(eng.volume_from_host(vol), np.linspace(0.5, 1.0, 22), MM_Y, MM_X, manifold=False)
    assert raw.faces.dtype == torch.int32
    check_smooth(eng, raw, PARAMS[2:4])
    sdf = VoxelProcessor().compute_sdf(vol, (0.7, MM_Y, MM_X))
    v, f = SurfaceExtractor().extract_surface_from_sdf(sdf, np.full(22, 0.7), MM_Y, MM_X, 0.0)
    check_smooth(eng, eng.mesh_from_host(v, f), PARAMS[3:4])


def host_mesh(rng, V, F, clusters):
    """Faces inside vertex clusters, degenerate and repeated faces, unreferenced vertices, zeros of both signs."""
    cl = rng.integers(0, clusters, V)
    f = np.concatenate([rng.choice(np.flatnonzero(cl == c), (F // clusters, 3)) for c in range(clusters) if (cl == c).any()])
    f = f[~(rng.random(V) < 0.1)[f].any(axis=1)]
    f = np.concatenate([f, f[:50], f[:20, [0, 0, 1]], f[:5, [1, 1, 1]]])
    v = (rng.standard_normal((V, 3)) * 50).astype(np.float32)
    v[rng.random((V, 3)) < 0.02] = -0.0
    v[rng.random((V, 3)) < 0.02] = 0.0
    return v, f


@gpu
@pytest.mark.parametrize("dtype", [np.int32, np.int64])
def test_host_meshes(eng, dtype):
    rng = np.random.default_rng(67)
    for V, F, k in ((5000, 6000, 40), (70000, 200000, 3), (300, 50, 300), (200, 3000, 2)):
        v, f = host_mesh(rng, V, F, k)
        check_smooth(eng, eng.mesh_from_host(v, f.astype(dtype)), PARAMS[1:4])


def fan(n, closed, rng):
    """n triangles around vertex 0: the hub's row has 2n raw entries (a face gives each of its vertices two raw entries or
    none, so raw rows have even lengths; 64 is the longest the warp sorts, 66 the shortest of the long-row path)."""
    i = np.arange(1, n + 1)
    f = np.stack([np.zeros(n, np.int64), i, (i % n) + 1 if closed else i + 1], axis=1)
    f = f[rng.permutation(n)]
    v = rng.standard_normal((n + 2, 3)).astype(np.float32)
    return v, f


@gpu
def test_rows_around_the_warp_limit_and_a_huge_fan(eng):
    rng = np.random.default_rng(71)
    for n, closed, want in ((32, True, 64), (32, False, 64), (33, True, 66), (33, False, 66), (200, True, 400)):
        v, f = fan(n, closed, rng)
        assert raw_row_lengths(f, len(v))[0] == want
        check_smooth(eng, eng.mesh_from_host(v, f), PARAMS[1:4])
    v, f = fan(100_000, False, rng)
    off, _ = check_smooth(eng, eng.mesh_from_host(v, f.astype(np.int32)), PARAMS[2:4])
    assert off[1] - off[0] == 100_001


@gpu
def test_empty_meshes(eng):
    import torch
    dev = torch.device("cuda")
    for V in (0, 4):
        for dt in (torch.int32, torch.int64):
            m = eng.DeviceMesh(torch.ones((V, 3), dtype=torch.float32, device=dev), torch.zeros((0, 3), dtype=dt, device=dev))
            off, nb = check_smooth(eng, m, PARAMS[:4])
            assert off.tolist() == [0] * (V + 1) and len(nb) == 0


@gpu
def test_repeated_runs_are_identical(eng):
    mesh = extracted(np.random.default_rng(73).random((30, 80, 100)) < 0.25)
    a1 = eng.vertex_neighbors(mesh)
    assert eng.vertex_neighbors(mesh) is a1
    fresh = eng.DeviceMesh(mesh.verts.clone(), mesh.faces.clone())
    a2 = eng.vertex_neighbors(fresh)
    assert a2 is not a1
    for x, y in zip(a1, a2):
        assert bits_equal(x.cpu().numpy(), y.cpu().numpy())
    assert bits_equal(eng.smooth_mesh(mesh).verts.cpu().numpy(), eng.smooth_mesh(fresh).verts.cpu().numpy())


@gpu
def test_smoothed_surface_through_the_registry_and_exporters(eng, phantom, tmp_path):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    from tomography_3d_reconstructor_b200.glb_exporter import glb_bytes, parse_glb
    from tomography_3d_reconstructor_b200.obj_exporter import OBJExporter
    se = SurfaceExtractor()
    v, f = se.extract_manifold_surface(phantom, np.linspace(0.4, 0.9, 24), MM_Y, MM_X)
    v2, f2 = se.smooth_surface(v, f)
    off, nb = so.adjacency(f, len(v))
    want = so.taubin(v, off, nb)
    assert bits_equal(v2, want) and bits_equal(f2, f)
    assert not v2.flags.writeable and not f2.flags.writeable
    mesh = eng.meshes.lookup(v2)
    assert mesh is not None and eng.meshes.lookup(f2) is mesh
    # smoothing the smoothed surface reuses its adjacency
    v3, f3 = se.smooth_surface(v2, f2, 4, 0.6, 0.6)
    assert eng.meshes.lookup(v3)._adjacency is mesh._adjacency
    assert bits_equal(v3, so.taubin(want, off, nb, 4, 0.6, 0.6))
    # measures, normals and bodies equal those of a fresh upload of the same arrays
    cv, cf = np.array(v2), np.array(f2)
    assert se.calculate_mesh_volume(v2, f2) == se.calculate_mesh_volume(cv, cf)
    assert se.calculate_surface_area(v2, f2) == se.calculate_surface_area(cv, cf) < se.calculate_surface_area(v, f)
    n2 = se.vertex_normals(v2, f2)             # area-weighted, summed with float atomics: equal up to rounding
    assert n2.shape == v2.shape and np.allclose(n2, se.vertex_normals(cv, cf), rtol=0, atol=1e-5)
    lab, n = se.split_surface(v2, f2)
    assert n == 1 and bits_equal(lab, bo.labels(f2, len(v2))[0])
    fv, ff = se.filter_surface_bodies(v2, f2, max_bodies=1)
    assert bits_equal(fv, v2) and bits_equal(ff, f2)
    pos, idx, _col, _doc = parse_glb(glb_bytes(v2, f2))
    assert bits_equal(pos, v2)
    assert np.array_equal(idx.astype(np.int64), f2) or np.array_equal(idx.astype(np.int64), f2[:, [0, 2, 1]])
    a, b = str(tmp_path / "a.obj"), str(tmp_path / "b.obj")
    assert OBJExporter().export_to_obj(v2, f2, a) and OBJExporter().export_to_obj(cv, cf, b)
    assert open(a, "rb").read() == open(b, "rb").read()
    # int32 faces keep their dtype
    v4, f4 = se.smooth_surface(np.array(v), np.array(f).astype(np.int32))
    assert f4.dtype == np.int32 and bits_equal(v4, want)


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
    check_smooth(eng, mesh)


@gpu
def test_refusals(eng):
    v = np.zeros((3, 3), np.float32)
    with pytest.raises(ValueError):
        eng.vertex_neighbors(eng.mesh_from_host(v, np.array([[0, 1, 3]])))
    with pytest.raises(ValueError):
        eng.vertex_neighbors(eng.mesh_from_host(v, np.array([[0, -1, 2]], np.int32)))
    mesh = eng.mesh_from_host(v, np.array([[0, 1, 2]]))
    for it, lamb, nu in ((-1, 0.5, 0.5), (2, float("nan"), 0.5), (2, 0.5, float("inf")), (2 ** 31, 0.5, 0.5)):
        with pytest.raises(ValueError):
            eng.smooth_mesh(mesh, it, lamb, nu)
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    with pytest.raises(ValueError):
        SurfaceExtractor().smooth_surface(v, np.array([[0, 1, 2]]), -3)


# ---- host only --------------------------------------------------------------------------------------------------------
def test_size_limits_are_refused_with_the_count():
    """Vertex counts beyond int32 and face counts beyond (2^32 - 1) / 6 (2^31 included) return status 2 naming the count,
    before any memory is touched; so do negative iterations and non-finite factors."""
    import os
    from tomography_3d_reconstructor_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    lib = _lib.load()
    n = 2 ** 31 + 5
    assert lib.t3d_mesh_adjacency_count(None, 0, 0, n, None, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
    assert lib.t3d_mesh_adjacency_count(None, 2 ** 31, 1, 10, None, None, None, None) == 2
    assert str(2 ** 31).encode() in lib.t3d_last_error()
    assert lib.t3d_mesh_adjacency_count(None, 715_827_883, 1, 10, None, None, None, None) == 2
    assert lib.t3d_mesh_adjacency_emit(n, 0, None, None, None, None) == 2
    assert lib.t3d_mesh_taubin(None, n, None, None, 1, 0.5, 0.5, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
    assert lib.t3d_mesh_taubin(None, 10, None, None, -1, 0.5, 0.5, None, None, None) == 2
    assert lib.t3d_mesh_taubin(None, 10, None, None, 1, float("nan"), 0.5, None, None, None) == 2
