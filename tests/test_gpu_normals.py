"""Field-gradient vertex normals (DESIGN.md §2) on the GPU against the numpy oracle (tests/normals_oracle.py), bit for bit:
the staged extraction, the SDF path, the fused step (staged first call, graph replay, generic sort), the geometry on a
convex phantom and the GLB NORMAL attribute."""
import numpy as np
import pytest
import torch

from conftest import random_blobs
import normals_oracle as no
from test_normals_oracle import MM, tie_field, volumes

pytestmark = pytest.mark.gpu

PHYS = (6.0, 143.1, 95.03)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def ragged():
    """The ragged shapes of test_gpu_shape_variants / the surface suite: W = 1, W one over a word or a uint4, one slice."""
    rng = np.random.default_rng(11)
    out = {}
    for name, shape in (("w1", (6, 9, 1)), ("w33", (5, 7, 33)), ("w129", (4, 6, 129)), ("z1", (1, 13, 17))):
        v = random_blobs(rng, shape, 0.5, 1.0)
        v[:, shape[1] // 2, :] = True
        out[name] = (v, np.linspace(0.2, 0.4, shape[0]), True)
    return out


def all_cases():
    c = dict(volumes())
    c.update(ragged())
    return c


@pytest.mark.parametrize("name", list(all_cases()))
def test_ex_normals_bit_equal_to_the_oracle(eng, oracle, name):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    vol, depths, add_padding = all_cases()[name]
    se = SurfaceExtractor()
    ref_v, ref_n = no.gradient_normals(vol, depths, MM[0], MM[1], True, add_padding)
    plain = se.extract_manifold_surface(vol, depths, MM[0], MM[1], True, True, add_padding)
    res = se.extract_manifold_surface_ex(vol, depths, MM[0], MM[1], True, True, add_padding)
    assert plain is not None and res is not None, se.last_error
    v, f, n = res
    assert np.array_equal(_bits(v), _bits(plain[0])) and np.array_equal(f, plain[1])
    assert np.array_equal(_bits(v), _bits(ref_v))
    assert n.dtype == np.float32 and not n.flags.writeable
    assert np.array_equal(_bits(n), _bits(ref_n))


def test_non_manifold_normals_follow_the_raw_order(eng, oracle):
    vol, depths, _ = volumes()["noise_ambiguous"]
    dv = eng.volume_from_host(vol)
    mesh = eng.extract_surface(dv, depths, MM[0], MM[1], False, True, normals=True)
    ref_v, ref_n = no.gradient_normals(vol, depths, MM[0], MM[1], False, True)
    assert np.array_equal(_bits(mesh.verts.cpu().numpy()), _bits(ref_v))
    assert np.array_equal(_bits(mesh.normals.cpu().numpy()), _bits(ref_n))


def _sdf_cases(oracle):
    vol = volumes()["ellipsoid_20_64_20"][0][30:70]
    sdf = oracle.signed_distance(vol, (0.1, MM[0], MM[1])).astype(np.float32)
    return {"ellipsoid_sdf": (sdf, 0.0, np.full(sdf.shape[0], 0.1)), "tie_field": tie_field() + (np.linspace(0.5, 1.5, 12),)}


@pytest.mark.parametrize("name", ["ellipsoid_sdf", "tie_field"])
def test_sdf_normals_bit_equal_to_the_dense_oracle(eng, oracle, name):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    f, level, depths = _sdf_cases(oracle)[name]
    se = SurfaceExtractor()
    res = se.extract_surface_from_sdf(f, depths, MM[0], MM[1], level, with_normals=True)
    assert res is not None, se.last_error
    v, faces, n = res
    uv, un, merged = no.gradient_normals_dense(f, level, depths, MM[0], MM[1])
    if name == "tie_field":
        assert merged == 5
    assert np.array_equal(_bits(v), _bits(uv)) and np.array_equal(_bits(n), _bits(un))
    plain = se.extract_surface_from_sdf(f, depths, MM[0], MM[1], level)
    assert len(plain) == 2 and np.array_equal(_bits(plain[0]), _bits(v)) and np.array_equal(plain[1], faces)


def _stack(Z=40, H=72, W=96):
    from oracle import cpu_ref
    u8 = cpu_ref.ellipsoid_phantom_u8(Z, H, W)
    return u8, [u8[z] >= 200 for z in range(Z)], (Z // 8, Z - 2 * (Z // 8), Z // 8)


def _reference_normals(oracle, u8, sides):
    ref = oracle.reference_pipeline(u8, 200, sides, *PHYS)
    Z, H, W = u8.shape
    depths = oracle.calculate_slice_depths(PHYS[0], *sides)
    v, n = no.gradient_normals(ref["smoothed"], depths, PHYS[2] / H, PHYS[1] / W, True, True)
    return ref, v, n


def _clear(pipeline):
    pipeline._plans.clear(); pipeline._hints.clear(); pipeline._g0_caps.clear(); pipeline._generic_sort.clear()


def test_fused_normals_staged_replay_and_generic_sort(eng, oracle):
    from tomography_3d_reconstructor_b200 import pipeline
    u8, masks, sides = _stack()
    ref, ref_v, ref_n = _reference_normals(oracle, u8, sides)
    _clear(pipeline)
    outs = [pipeline.reconstruct_host(masks, 1, sides, *PHYS, normals=True) for _ in range(3)]   # staged, capture, replay
    key = pipeline.plan_key(pipeline._device_inputs[((u8.shape), torch.cuda.current_device())], 1, sides, *PHYS, normals=True)
    assert key in pipeline._plans and pipeline._plans[key].graph is not None
    for out in outs:
        assert np.array_equal(_bits(out["vertices"]), _bits(ref_v)) and np.array_equal(out["faces"], ref["faces"])
        assert np.array_equal(_bits(out["normals"]), _bits(ref_n))
    # the generic 64-bit sort instead of the structured ordering
    pipeline._generic_sort[key] = True
    pipeline._plans.pop(key, None)
    for _ in range(2):
        out = pipeline.reconstruct_host(masks, 1, sides, *PHYS, normals=True)
        assert pipeline._plans[key].caps[3] == 0
        assert np.array_equal(_bits(out["vertices"]), _bits(ref_v)) and np.array_equal(_bits(out["normals"]), _bits(ref_n))
    # the staged path with its own unverified-order fallback (generic canonicalisation): forced through set_sizes
    dv = eng.volume_from_host(ref["smoothed"])
    depths = oracle.calculate_slice_depths(PHYS[0], *sides)
    m = eng.extract_surface(dv, depths, PHYS[2] / u8.shape[1], PHYS[1] / u8.shape[2], True, True, canonical="async", normals=True)
    m.set_sizes(0, 0, 1)
    assert np.array_equal(_bits(m.normals.cpu().numpy()), _bits(ref_n))
    _clear(pipeline)


def test_fused_without_normals_is_unchanged(eng, oracle):
    from tomography_3d_reconstructor_b200 import _lib, pipeline
    u8, masks, sides = _stack(32, 64, 80)
    ref = oracle.reference_pipeline(u8, 200, sides, *PHYS)
    _clear(pipeline)
    for _ in range(3):
        out = pipeline.reconstruct_host(masks, 1, sides, *PHYS)
        assert "normals" not in out
        assert np.array_equal(out["vertices"], ref["vertices"]) and np.array_equal(out["faces"], ref["faces"])
    for _ in range(2):
        pipeline.reconstruct_host(masks, 1, sides, *PHYS, normals=True)
    buf = pipeline._device_inputs[((u8.shape), torch.cuda.current_device())]
    L = _lib.load()
    counts = []
    for normals in (False, True):
        plan = pipeline._plans[pipeline.plan_key(buf, 1, sides, *PHYS, normals=normals)]
        torch.cuda.synchronize()
        c0 = L.t3d_launch_count()
        plan.enqueue(buf)
        counts.append(L.t3d_launch_count() - c0)
        torch.cuda.synchronize()
    assert counts[1] == counts[0] + 2       # the plain step is t3d_reconstruct alone; normals add the tie pass + the kernel
    plain = pipeline._plans[pipeline.plan_key(buf, 1, sides, *PHYS)]
    assert plain.normals is None
    _clear(pipeline)


def test_normals_geometry_on_the_convex_phantom(eng, oracle):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    vol = oracle.smooth_voxel_data(oracle.ellipsoid_phantom_u8(48, 80, 96) >= 200, 3, True)
    depths = oracle.calculate_slice_depths(6.0, 6, 36, 6)
    se = SurfaceExtractor()
    v, f, n = se.extract_manifold_surface_ex(vol, depths, MM[0], MM[1])
    v64, n64 = v.astype(np.float64), n.astype(np.float64)
    centre = 0.5 * (v64.min(axis=0) + v64.max(axis=0))
    assert np.all(np.einsum("ij,ij->i", n64, v64 - centre) > 0)
    assert np.all(np.abs(np.linalg.norm(n64, axis=1) - 1) <= 1e-6)
    # the area-weighted normals follow the face winding, which points into the object in the [z, y, x] column order (a
    # reflection of x, y, z): compare with them turned outwards
    a = -se.vertex_normals(v, f).astype(np.float64)
    cos = np.einsum("ij,ij->i", n64, a) / np.maximum(np.linalg.norm(a, axis=1), 1e-30)
    assert (cos >= 0.9).mean() >= 0.99


def test_glb_normal_attribute_round_trips(eng, oracle, tmp_path):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor
    from tomography_3d_reconstructor_b200.glb_exporter import GLBExporter, glb_bytes, parse_glb
    vol = oracle.smooth_voxel_data(oracle.ellipsoid_phantom_u8(24, 56, 72) >= 200, 3, True)
    depths = oracle.calculate_slice_depths(6.0, 3, 18, 3)
    se, ex = SurfaceExtractor(), GLBExporter()
    v, f, n = se.extract_manifold_surface_ex(vol, depths, 0.3, 0.25)
    path = str(tmp_path / "model.glb")
    for faces in (f, f[:, [0, 2, 1]].copy()):       # as extracted, and inside out (the writer flips the winding)
        assert ex.export_to_glb(v, faces, path, None, n) is True
        data = open(path, "rb").read()
        pos, idx, col, nrm, doc = parse_glb(data, with_normals=True)
        assert col is None and np.array_equal(_bits(pos), _bits(v)) and np.array_equal(_bits(nrm), _bits(n))
        assert "NORMAL" in doc["meshes"][0]["primitives"][0]["attributes"] and len(data) % 4 == 0
        p64 = pos.astype(np.float64)
        a, b, c = p64[idx[:, 0]], p64[idx[:, 1]], p64[idx[:, 2]]
        assert np.einsum("ij,ij->i", a, np.cross(b, c)).sum() > 0
    colors = ex.create_layer_colors(v, depths, 3, 20, 1.0)
    pos, idx, col, nrm, doc = parse_glb(glb_bytes(v, f, colors, n), with_normals=True)
    assert np.array_equal(col, colors) and np.array_equal(_bits(nrm), _bits(n))
    # without normals: the same bytes as a file written without the argument, and no NORMAL attribute
    assert glb_bytes(v, f, colors) == glb_bytes(v, f, colors, None)
    assert parse_glb(glb_bytes(v, f), with_normals=True)[3] is None
    with pytest.raises(ValueError):
        glb_bytes(v, f, None, n.astype(np.float64))
