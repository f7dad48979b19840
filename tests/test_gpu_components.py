"""Connected components on the device (csrc/t3d_label.cu) against scipy.ndimage.label, find_objects and the reference's own
volume / bounding-box functions applied to each component alone, bit for bit; the component filter against np.isin."""
import numpy as np
import pytest
from scipy import ndimage

from conftest import random_blobs

gpu = pytest.mark.gpu

STRUCT = {6: ndimage.generate_binary_structure(3, 1), 26: np.ones((3, 3, 3), bool)}
MM_X, MM_Y = 0.37, 0.29


def scipy_label(vol, conn):
    lab, k = ndimage.label(vol, STRUCT[conn])
    return lab, k


def noise(rng, shape, density):
    return rng.random(shape) < density


def serpentine(Z, H, W):
    """One component through every row and plane: full rows at even y, one end voxel at odd y alternating sides; odd planes
    hold one voxel joining the planes either side, alternately at the first and the last corner."""
    v = np.zeros((Z, H, W), bool)
    for z in range(0, Z, 2):
        v[z, 0::2, :] = True
        for y in range(1, H, 2):
            v[z, y, W - 1 if (y // 2) % 2 == 0 else 0] = True
    for z in range(1, Z, 2):
        v[z, 0, 0] = (z % 4 == 1)
        v[z, H - 1, W - 1] = (z % 4 == 3)
    return v


def comb(Z, H, W):
    """Teeth every other x, separate in every plane but the last, which joins them."""
    v = np.zeros((Z, H, W), bool)
    v[:, :, 0::2] = True
    v[-1] = True
    return v


def checkerboard(Z, H, W):
    z, y, x = np.indices((Z, H, W))
    return (z + y + x) % 2 == 0


def cases():
    rng = np.random.default_rng(2026)
    from oracle import cpu_ref
    c = {}
    for d in (0.05, 0.3, 0.5, 0.9):
        c["noise%.2f" % d] = noise(rng, (23, 45, 71), d)
    c["blobs"] = random_blobs(rng, (30, 50, 90), 0.4, 1.5)
    c["phantom"] = cpu_ref.ellipsoid_phantom_u8(24, 64, 96) >= 200
    c["empty"] = np.zeros((5, 7, 33), bool)
    c["full"] = np.ones((5, 7, 33), bool)
    c["checker"] = checkerboard(6, 9, 37)
    c["serpentine"] = serpentine(9, 15, 40)
    c["comb"] = comb(7, 11, 65)
    return c


CASES = cases()


@gpu
@pytest.mark.parametrize("conn", [6, 26])
@pytest.mark.parametrize("name", list(CASES))
def test_labels_equal_scipy(eng, name, conn):
    from tomography_3d_reconstructor_b200 import VoxelProcessor
    vol = CASES[name]
    lab, k = VoxelProcessor().label_components(vol, conn)
    ref, rk = scipy_label(vol, conn)
    assert lab.dtype == np.int32 and lab.shape == vol.shape
    assert k == rk and np.array_equal(lab, ref)
    if name == "phantom" or name == "full":
        assert k == 1
    if name == "empty":
        assert k == 0
    if name == "checker":
        assert k == (int(vol.sum()) if conn == 6 else 1)
    if name in ("serpentine", "comb"):
        assert k == 1


@gpu
@pytest.mark.parametrize("conn", [6, 26])
def test_labels_on_shapes_crossing_word_and_row_boundaries(eng, conn):
    from tomography_3d_reconstructor_b200 import VoxelProcessor
    vp = VoxelProcessor()
    rng = np.random.default_rng(7)
    for W in (1, 31, 32, 33, 129, 300):
        for H in (1, 7, 64):
            for Z in (1, 5, 40):
                vol = noise(rng, (Z, H, W), 0.45)
                lab, k = vp.label_components(vol, conn)
                ref, rk = scipy_label(vol, conn)
                assert k == rk and np.array_equal(lab, ref), (Z, H, W)


@gpu
@pytest.mark.parametrize("conn", [6, 26])
def test_labels_large_noise_at_the_percolation_threshold(eng, conn):
    """128 x 512 x 512 at density 0.3: ~2 M components at 6, one giant tortuous component at 26."""
    from tomography_3d_reconstructor_b200 import VoxelProcessor
    vol = noise(np.random.default_rng(3), (128, 512, 512), 0.3)
    lab, k = VoxelProcessor().label_components(vol, conn)
    ref, rk = scipy_label(vol, conn)
    assert k == rk and np.array_equal(lab, ref)


@gpu
def test_grids_from_the_package_are_labelled_without_upload(eng, oracle, monkeypatch):
    from tomography_3d_reconstructor_b200 import VoxelProcessor
    Z, H, W = 16, 40, 100                        # W not a multiple of 32
    rng = np.random.default_rng(5)
    masks = list(random_blobs(rng, (Z, H, W), 0.35, 1.2))
    vp = VoxelProcessor()
    vox = vp.create_voxel_data(masks, True)
    sm = vp.smooth_voxel_data(vox, 3, True)
    for arr in (vox, sm):
        assert eng.volumes.lookup(arr) is not None

    def no_upload(*_a, **_k):
        raise AssertionError("a package grid was uploaded again")

    monkeypatch.setattr(eng, "upload_u8", no_upload)
    for arr in (vox, sm):
        for conn in (6, 26):
            lab, k = vp.label_components(arr, conn)
            ref, rk = scipy_label(np.asarray(arr), conn)
            assert k == rk and np.array_equal(lab, ref)


def volume_oracle(labels, K, mm_x, mm_y, slice_depths):
    """Per-(label, z) counts, then the float64 additions of volume_calculator.py:23-35 over ascending z for every label at
    once (the same operations in the same order as the reference's loop on labels == c)."""
    out = np.zeros(K + 1, dtype=np.float64)
    if len(slice_depths) == 0:
        return out[1:]
    for z in range(min(labels.shape[0], len(slice_depths))):
        c = np.bincount(labels[z].ravel(), minlength=K + 1)
        nz = np.flatnonzero(c[1:]) + 1
        out[nz] += c[nz] * (mm_x * mm_y * slice_depths[z])
    return out[1:]


@gpu
@pytest.mark.parametrize("conn", [6, 26])
@pytest.mark.parametrize("depths", ["full", "short", "empty"])
def test_stats_equal_the_reference_per_component(eng, oracle, conn, depths):
    from tomography_3d_reconstructor_b200 import VolumeCalculator
    rng = np.random.default_rng(11)
    vol = random_blobs(rng, (26, 48, 77), 0.3, 1.2) | noise(rng, (26, 48, 77), 0.02)
    Z = vol.shape[0]
    sd = {"full": np.linspace(0.4, 1.3, Z), "short": np.linspace(0.5, 0.9, Z - 9), "empty": np.array([])}[depths]
    res = VolumeCalculator().analyze_components(vol, MM_X, MM_Y, sd, conn)
    ref, K = scipy_label(vol, conn)
    assert res["n_components"] == K and K > 20
    assert res["voxel_counts"].dtype == np.int64 and np.array_equal(res["voxel_counts"], np.bincount(ref.ravel())[1:])
    objs = ndimage.find_objects(ref)
    box = np.array([[s.start if k % 2 == 0 else s.stop - 1 for s in o for k in (0, 1)] for o in objs], dtype=np.int32)
    assert res["bbox_index"].dtype == np.int32 and np.array_equal(res["bbox_index"], box)
    vol_ref = volume_oracle(ref, K, MM_X, MM_Y, sd)
    assert res["volume_mm3"].dtype == np.float64
    assert np.array_equal(res["volume_mm3"].view(np.uint64), vol_ref.view(np.uint64))
    largest = int(np.argmax(res["voxel_counts"])) + 1
    for c in list(range(1, 21)) + [largest]:
        one = ref == c
        v = oracle.calculate_voxel_volume_variable_depth(one, MM_X, MM_Y, sd)
        assert np.float64(v).view(np.uint64) == res["volume_mm3"][c - 1].view(np.uint64), c
        try:
            bb = oracle.calculate_bounding_box_variable_depth(one, MM_X, MM_Y, sd)
        except IndexError:                       # the component starts beyond the given depths: NaN there
            assert np.isnan(res["bbox_mm"][c - 1, :2]).all() and np.isnan(res["dimensions_mm"][c - 1, 2])
            continue
        got = res["bbox_mm"][c - 1]
        want = np.array([bb["z"][0], bb["z"][1], bb["y"][0], bb["y"][1], bb["x"][0], bb["x"][1]], dtype=np.float64)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), c
        assert np.array_equal(res["dimensions_mm"][c - 1].view(np.uint64), np.array(bb["dimensions"], np.float64).view(np.uint64))


@gpu
def test_filter_equals_isin(eng):
    from tomography_3d_reconstructor_b200 import VoxelProcessor
    vp = VoxelProcessor()
    rng = np.random.default_rng(13)
    vol = random_blobs(rng, (20, 40, 70), 0.3, 1.2) | noise(rng, (20, 40, 70), 0.03)
    vol[2:4, 2:4, 60:62] = True                  # two 8-voxel cubes: a tie in size
    vol[2:4, 30:32, 60:62] = True
    for conn in (6, 26):
        ref, K = scipy_label(vol, conn)
        counts = np.bincount(ref.ravel())[1:]
        for mv, mc in ((1, None), (2, None), (8, None), (50, None), (1, 1), (1, 3), (8, 2), (10 ** 9, None)):
            got = vp.filter_components(vol, min_voxels=mv, max_components=mc, connectivity=conn)
            kept = eng.component_keep(counts, mv, mc)
            assert got.dtype == np.bool_ and np.array_equal(got, np.isin(ref, kept)), (conn, mv, mc)
        largest = np.isin(ref, [int(np.argmax(counts)) + 1])
        assert np.array_equal(vp.filter_components(vol, max_components=1, connectivity=conn), largest)
    # the two equal cubes: keep-one keeps the earlier in raster order
    two = np.zeros((4, 34, 64), bool)
    two[2:4, 2:4, 60:62] = True
    two[2:4, 30:32, 60:62] = True
    lab, _ = scipy_label(two, 6)
    assert np.array_equal(vp.filter_components(two, max_components=1), lab == 1)
    for bad in ({"min_voxels": 0}, {"max_components": 0}, {"connectivity": 18}):
        with pytest.raises(ValueError):
            vp.filter_components(vol, **bad)
    with pytest.raises(ValueError):
        vp.label_components(vol, 8)


@gpu
def test_filter_smooth_extract_through_the_identity_cache(eng, oracle):
    from tomography_3d_reconstructor_b200 import SurfaceExtractor, VoxelProcessor, VolumeCalculator
    Z, H, W = 18, 48, 80
    vol = oracle.ellipsoid_phantom_u8(Z, H, W) >= 200
    rng = np.random.default_rng(17)
    vol |= noise(rng, (Z, H, W), 0.01)           # islands next to the object
    vp, se, vc = VoxelProcessor(), SurfaceExtractor(), VolumeCalculator()
    f = vp.filter_components(vol, max_components=1)
    ref_lab, _ = scipy_label(vol, 6)
    ref_f = np.isin(ref_lab, [int(np.argmax(np.bincount(ref_lab.ravel())[1:])) + 1])
    assert np.array_equal(f, ref_f) and eng.volumes.lookup(f) is not None
    sm = vp.smooth_voxel_data(f, 3, True)
    assert np.array_equal(sm, oracle.smooth_voxel_data(ref_f, 3, True))
    depths = np.linspace(0.3, 0.6, Z)
    v, fc = se.extract_manifold_surface(sm, depths, 0.2, 0.3, True, True, True)
    rv, rf = oracle.extract_manifold_surface(oracle.smooth_voxel_data(ref_f, 3, True), depths, 0.2, 0.3, True, True, True)
    assert v.shape == rv.shape and np.allclose(v, rv, rtol=1e-5, atol=1e-5) and np.array_equal(fc, rf)
    assert vc.calculate_voxel_volume_variable_depth(f, 0.3, 0.2, depths) == \
        oracle.calculate_voxel_volume_variable_depth(ref_f, 0.3, 0.2, depths)


@gpu
@pytest.mark.parametrize("conn", [6, 26])
def test_repeated_labelling_is_identical(eng, conn):
    """The atomic merge order must not show: a fresh labelling of the same grid gives the same arrays."""
    vol = noise(np.random.default_rng(19), (40, 96, 150), 0.3)
    outs = []
    for _ in range(2):
        dv = eng.volume_from_host(vol.copy())     # a new device volume: nothing memoised
        comps = eng.label_components(dv, conn)
        outs.append((comps.labels().cpu().numpy(), comps.counts().copy(), comps.bbox_index().copy(),
                     comps.volumes_mm3(MM_X, MM_Y, np.linspace(0.5, 1.0, 40))))
    for a, b in zip(*outs):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


# ---- host only --------------------------------------------------------------------------------------------------------
def test_component_keep_threshold_top_k_and_ties():
    from tomography_3d_reconstructor_b200.engine import component_keep
    counts = np.array([5, 1, 9, 5, 9, 2, 5], dtype=np.int64)          # labels 1..7
    assert component_keep(counts).tolist() == [1, 2, 3, 4, 5, 6, 7]
    assert component_keep(counts, 5).tolist() == [1, 3, 4, 5, 7]
    assert component_keep(counts, 6).tolist() == [3, 5]
    assert component_keep(counts, 10).tolist() == []
    assert component_keep(counts, max_components=1).tolist() == [3]            # tie 9 / 9: the lower label
    assert component_keep(counts, max_components=3).tolist() == [1, 3, 5]      # then 5 / 5 / 5: label 1
    assert component_keep(counts, 2, max_components=5).tolist() == [1, 3, 4, 5, 7]
    assert component_keep(counts, 1, max_components=100).tolist() == [1, 2, 3, 4, 5, 6, 7]
    assert component_keep(np.zeros(0, np.int64), max_components=1).tolist() == []
    for bad in ({"min_voxels": 0}, {"min_voxels": -3}, {"max_components": 0}):
        with pytest.raises(ValueError):
            component_keep(counts, **bad)


def test_run_and_component_limits_are_refused_with_the_count():
    """Beyond int32 runs the label call returns status 2 naming the count, before it touches any memory."""
    import os
    from tomography_3d_reconstructor_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    lib = _lib.load()
    n = 2 ** 31 + 5
    assert lib.t3d_cc_label(None, 4, 4, 4, 6, None, n, None, None, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
    assert lib.t3d_cc_label(None, 4, 4, 4, 18, None, 10, None, None, None, None, None) == 2
    assert lib.t3d_cc_stats(None, None, n, 4, 3, None, None, None) == 2
    assert str(n).encode() in lib.t3d_last_error()
