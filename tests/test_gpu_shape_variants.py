"""GPU parity of the kernel variants that only the shape of a volume selects, against the oracle.

Three variants carry the wide / large configurations and never run on the small shapes of the other suites:
  * k_morph4 (csrc/t3d_voxel.cu): opening + closing in one pass, fused single-device and slab steps with W in
    {512, 1024, 2048, 4096}; tiled in bands of `ty` rows and chunks of `zc` planes, 128-voxel uint4 columns;
  * the cp.async.bulk tile ring of k_sdf_envelope (csrc/t3d_edt.cu): y pass when W % 128 == 0, z pass when H * W % 8 == 0;
  * k_zsort_layers<8> (csrc/t3d_surface.cu), the batched-fetch layer sort: cap_z >= 4096 planes of the sign volume.
The shapes below are chosen to cross the tile boundaries of each variant; small mirrors of the host-side rules check that
every parameter set really reaches the variant (and its boundaries), so a later retune cannot quietly shrink the coverage.
The fused paths silently fall back to the staged path when a step overflows or fails its order check, so the tests also
assert that the fused plan produced the result.
"""
import functools

import numpy as np
import pytest
import torch

from conftest import random_blobs
from test_gpu_edt import _emulated_all_to_all, dev_volume

pytestmark = pytest.mark.gpu

PHYS = (6.0, 143.1, 95.03)
THRESHOLD = 200
MAX_CTAS_PER_SM = 16        # 2048 resident threads per SM / 128-thread CTAs: the most any occupancy allows


def _sides(Z):
    return (Z // 8, Z - 2 * (Z // 8), Z // 8)


def _sm_count():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ----------------------------------------------------------------------------------------------------------------
# mirrors of the host-side selection rules
# ----------------------------------------------------------------------------------------------------------------
def morph4_eligible(Z, H, W):
    """t3d_morph4_eligible (csrc/t3d_voxel.cu)."""
    return W % 128 == 0 and 512 <= W <= 4096 and 32 % (W // 128) == 0 and Z >= 1 and H >= 1


def morph4_tile(H, W, nz, sms):
    """(ty, zc): band height and planes per chunk that t3d_morph4_launch (csrc/t3d_voxel.cu) picks with its cost model for
    `nz` output planes on a device with `sms` multiprocessors."""
    M4_R, M4_PF = 2, 4
    nw4 = W // 128
    nw = 4 * nw4
    warp_rows = M4_R * (32 // nw4)
    rows_max = min(512 // nw4 * M4_R, (200 * 1024) // ((M4_PF + 6) * nw * 4))
    rows_max -= rows_max % warp_rows
    best, pick = float("inf"), None
    rr = rows_max
    while rr >= 16 and rr >= warp_rows:
        ty = rr - 8
        bands = -(-H // ty)
        per_sm = min(512 // (rr // M4_R * nw4), (220 * 1024) // ((M4_PF + 6) * rr * nw * 4))
        if per_sm >= 1:
            for c in (16, 24, 32, 48, 64, 96, 128):
                ctas = bands * -(-nz // c)
                load = -(-ctas // sms) * rr
                floor_ = 48.0 * -(-ctas // (sms * per_sm))
                cost = max(load, floor_) * (c + 8)
                if cost < best:
                    best, pick = cost, (ty, c)
        rr -= warp_rows
    return pick


def sdf_bulk_ok(off_a, off_b, n_lines, inner, outer_stride, stride):
    """sdf_bulk_ok (csrc/t3d_edt.cu); off_a / off_b: byte offsets of the two inputs from a 256-byte aligned allocation."""
    if off_a % 16 or off_b % 16 or stride % 8 or outer_stride % 8:
        return False
    if inner % 128 and outer_stride not in (0, inner):
        return False
    return (n_lines % 128) % 8 == 0


def sdf_bulk_passes(Z, H, W):
    """(y pass, z pass) of t3d_sdf on a (Z, H, W) volume run in bulk mode: the y pass reads the x-pass scratch (256-byte
    aligned) along lines (z, x); the z pass reads dy and dx = dy + Z*H*W int16 along lines (y, x)."""
    return (sdf_bulk_ok(0, 0, Z * W, W, H * W, W),
            sdf_bulk_ok(0, 2 * Z * H * W, H * W, H * W, 0, H * W))


def zsort_batched(cap_z, Zs):
    """k_zsort_layers<8> instead of <1> (t3d_mesh_canonicalize_structured_dev, csrc/t3d_surface.cu); Zs = planes of the
    padded sign volume the step marches."""
    return cap_z >= 4096 * Zs


# ----------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------
def _clear_plans():
    from tomography_3d_reconstructor_b200 import pipeline
    pipeline._plans.clear(); pipeline._hints.clear(); pipeline._g0_caps.clear(); pipeline._generic_sort.clear()


def _only_plan():
    from tomography_3d_reconstructor_b200 import pipeline
    assert len(pipeline._plans) == 1
    return next(iter(pipeline._plans.values()))


def _fused_from_plan(out):
    """Asserts that reconstruct_fused returned the fused plan's result (not a staged fallback) and returns the plan."""
    from tomography_3d_reconstructor_b200 import pipeline
    plan = _only_plan()
    assert out["mesh"].verts.data_ptr() == plan.verts.data_ptr(), "served by the staged fallback"
    assert plan.caps[3] > 0, "structured ordering not provisioned"
    assert not pipeline._generic_sort, "the structured vertex order was rejected and the step re-run with the generic sort"
    h = plan.res_np
    assert h[pipeline.R_OVERFLOW] == 0 and h[pipeline.R_UNVERIFIED] == 0
    return plan


def _assert_matches_oracle(out, ref, plan, Z):
    from tomography_3d_reconstructor_b200 import pipeline
    v, f = out["mesh"].verts.cpu().numpy(), out["mesh"].faces.cpu().numpy()
    assert v.shape == ref["vertices"].shape and f.shape == ref["faces"].shape
    assert np.array_equal(v.view(np.uint32), ref["vertices"].view(np.uint32))
    assert np.array_equal(f, ref["faces"])
    # the per-plane counts the step accumulates (smoothed: by k_morph4 / the last k_morph stage), then the volumes
    counts = plan.res_np[pipeline.R_COUNTS:pipeline.R_COUNTS + 2 * Z].reshape(2, Z)
    assert np.array_equal(counts[0], ref["voxel_data"].sum(axis=(1, 2)))
    assert np.array_equal(counts[1], ref["smoothed"].sum(axis=(1, 2)))
    assert out["voxel_volume_mm3"] == ref["voxel_volume"]
    assert out["processed_voxel_volume_mm3"] == ref["processed_volume"]


def _box(occ, z, y, x):
    """occ[z0:z1, y0:y1, x0:x1] = True, clipped to the volume."""
    Z, H, W = occ.shape
    (z0, z1), (y0, y1), (x0, x1) = z, y, x
    occ[max(z0, 0):min(z1, Z), max(y0, 0):min(y1, H), max(x0, 0):min(x1, W)] = True


def built_volume(Z, H, W, ty, zc):
    """Hand-placed features on the k_morph4 tile boundaries: 1- and 3-voxel plates (opening removes / keeps them),
    one-voxel gaps and holes (closing fills them), objects touching all six faces, features across the uint4 columns
    (x = 128 k - 1 | 128 k), the bands (y = ty - 1 | ty | ty + 1, y = H - 1) and the chunks (z = zc - 1 | zc, z = Z - 1)."""
    occ = np.zeros((Z, H, W), bool)
    # the six faces
    _box(occ, (0, Z), (0, 3), (20, 60))                 # y = 0, z = 0 and z = Z-1
    _box(occ, (0, Z), (H - 2, H), (70, 110))            # y = H-1 (two rows)
    _box(occ, (2, Z - 2), (10, 30), (0, 4))             # x = 0
    _box(occ, (2, Z - 2), (10, 30), (W - 4, W))         # x = W-1
    _box(occ, (Z - 1, Z), (5, 25), (300, 340))          # a lone one-plane object at z = Z-1
    # across every uint4 column boundary b = 128 k
    for k, b in enumerate(range(128, W, 128)):
        g = b - 1 if k % 2 == 0 else b                  # one-voxel gap at x = 127 | 128, 255 | 256, ...
        _box(occ, (zc - 3, zc + 3), (ty - 3, ty + 3), (g - 6, g))
        _box(occ, (zc - 3, zc + 3), (ty - 3, ty + 3), (g + 1, g + 7))
        _box(occ, (1, Z - 1), (5, 12), (b, b + 1))      # 1-voxel plate on the first voxel of a column
        _box(occ, (1, Z - 1), (14, 22), (b - 1, b + 2))  # 3-voxel plate across the boundary
        _box(occ, (3, Z - 3), (H - 8, H), (b - 2, b + 2))   # touches y = H-1 across the boundary
    # across the band boundary: gaps at y = ty - 1, ty, ty + 1, a one-row line at y = ty
    for i, gy in enumerate((ty - 1, ty, ty + 1)):
        x0 = 150 + 40 * i
        _box(occ, (2, Z - 2), (gy - 5, gy), (x0, x0 + 30))
        _box(occ, (2, Z - 2), (gy + 1, gy + 6), (x0, x0 + 30))
    _box(occ, (2, Z - 2), (ty, ty + 1), (280, 296))
    # across the chunk boundary: gaps at z = zc - 1 and zc, a 3-plane plate, a 1-plane plate
    _box(occ, (zc - 5, zc - 1), (24, 34), (350, 380)); _box(occ, (zc, zc + 4), (24, 34), (350, 380))
    _box(occ, (zc - 4, zc), (24, 34), (390, 420)); _box(occ, (zc + 1, zc + 5), (24, 34), (390, 420))
    _box(occ, (zc - 1, zc + 2), (2, 20), (430, 470))
    _box(occ, (zc, zc + 1), (22, 30), (430, 470))
    # a solid block across a band, a chunk and a column boundary with single-voxel holes on all three
    _box(occ, (3, Z - 1), (ty - 6, ty + 6), (100, 160))
    for z in (zc - 1, zc, 5):
        for y in (ty - 1, ty, ty + 1):
            for x in (127, 128, 140):
                if 3 < z < Z - 2 and y < H - 1:
                    occ[z, y, x] = False
    return occ


def _blobs_u8(shape, sigma, seed, density=0.5):
    return (random_blobs(np.random.default_rng(seed), shape, density, sigma) * 255).astype(np.uint8)


# content and oracle results are shared by the tests that use the same volume
@functools.lru_cache(maxsize=None)
def _volume(kind, shape):
    Z, H, W = shape
    if kind == "blobs_s1":
        return _blobs_u8(shape, 1.0, Z * W + H)
    if kind == "blobs_s2":
        return _blobs_u8(shape, 2.0, Z * W + H + 1)
    if kind == "built":
        ty, zc = morph4_tile(H, W, Z, 148)
        return (built_volume(Z, H, W, ty, zc) * 255).astype(np.uint8)
    if kind == "holes":
        return ((np.random.default_rng(W).random(shape) < 0.9) * 255).astype(np.uint8)
    if kind == "ellipsoid":
        from oracle import cpu_ref
        u8 = cpu_ref.ellipsoid_phantom_u8(Z, H, W)
        u8[0, H // 2 - 2:H // 2 + 2, W // 2 - 3:W // 2 + 3] = 0
        return u8
    if kind == "plate":
        u8 = np.zeros(shape, np.uint8)
        u8[Z // 3:Z // 3 + 4] = 255               # spans the whole image: long runs of equal z keys
        return u8
    raise ValueError(kind)


@functools.lru_cache(maxsize=None)
def _reference(kind, shape):
    from oracle import cpu_ref
    return cpu_ref.reference_pipeline(_volume(kind, shape), THRESHOLD, _sides(shape[0]), *PHYS)


# ----------------------------------------------------------------------------------------------------------------
# 1. k_morph4 against the oracle
# ----------------------------------------------------------------------------------------------------------------
MORPH4_CASES = [((17, 41, W), "blobs_s1") for W in (512, 1024, 2048, 4096)] + \
               [((20, 50, W), kind) for W in (512, 1024, 2048, 4096) for kind in ("blobs_s2", "built")]
MORPH4_TINY = ((2, 3, 512), "holes")


def test_morph4_shapes_cross_bands_and_chunks():
    """Every k_morph4 shape is eligible and spans >= 2 bands and >= 2 z-chunks of the tile the cost model picks; the pick
    does not depend on the SM count for grids this small."""
    for (Z, H, W), _kind in MORPH4_CASES + [MORPH4_TINY]:
        assert morph4_eligible(Z, H, W)
        picks = {morph4_tile(H, W, Z, sms) for sms in (100, 132, 148, 160, 264)}
        assert len(picks) == 1
    for (Z, H, W), _kind in MORPH4_CASES:
        ty, zc = morph4_tile(H, W, Z, 148)
        assert (ty, zc) == ((24 if W == 4096 else 40), 16)
        assert -(-H // ty) >= 2 and -(-Z // zc) >= 2, ((Z, H, W), ty, zc)
    assert {W for (_z, _h, W), _k in MORPH4_CASES} == {512, 1024, 2048, 4096}
    assert not morph4_eligible(20, 50, 384)


@pytest.mark.parametrize("shape,kind", MORPH4_CASES + [MORPH4_TINY], ids=lambda p: "x".join(map(str, p)) if isinstance(p, tuple) else p)
def test_morph4_fused_step_matches_the_oracle(eng, oracle, shape, kind):
    """The fused single-device step on wide rows (k_morph4 + the one-pass pack) against reference_pipeline: identical
    mesh, exact per-plane raw / smoothed counts; the fused plan (not the staged fallback) produced the result."""
    from tomography_3d_reconstructor_b200 import pipeline
    Z, H, W = shape
    u8 = _volume(kind, shape)
    ref = _reference(kind, shape)
    assert ref.get("vertices") is not None and len(ref["faces"]) > 0
    if kind != "holes":       # opening / closing really change these volumes
        assert (ref["smoothed"] != ref["voxel_data"]).sum() > 100
    masks = torch.from_numpy(u8).cuda()
    args = (THRESHOLD, _sides(Z), *PHYS)
    _clear_plans()
    pipeline.reconstruct_fused(masks, *args, use_graph=False)          # staged: learns the sizes
    # fused: the first step may provision the clamp-group sort and re-run, and the sizes it reports may exceed the staged
    # step's and raise the hints once, so the plan can be rebuilt once; then it stays
    plans = []
    for rep in range(3):
        out = pipeline.reconstruct_fused(masks, *args, use_graph=False)
        plans.append(_fused_from_plan(out))
        _assert_matches_oracle(out, ref, plans[-1], Z)
    assert plans[2] is plans[1], "no steady state"


def test_morph4_replaces_the_four_launch_chain(eng, oracle):
    """Launch count of one eager fused step: the same content at W = 384 (one-pass pack, four-launch k_morph chain) and
    zero-padded to W = 512 (k_morph4) differs by exactly the three saved morphology launches."""
    from tomography_3d_reconstructor_b200 import _lib, pipeline
    lib = _lib.load()
    Z, H = 20, 50
    narrow = _blobs_u8((Z, H, 384), 1.5, 11)
    wide = np.zeros((Z, H, 512), np.uint8)
    wide[:, :, :384] = narrow
    assert not morph4_eligible(Z, H, 384) and morph4_eligible(Z, H, 512)
    args = (THRESHOLD, _sides(Z), *PHYS)
    launches = {}
    for u8 in (narrow, wide):
        masks = torch.from_numpy(u8).cuda()
        _clear_plans()
        for _ in range(3):                        # staged (learns), fused (may re-plan once), steady state
            pipeline.reconstruct_fused(masks, *args, use_graph=False)
        torch.cuda.synchronize()
        n0 = lib.t3d_launch_count()
        out = pipeline.reconstruct_fused(masks, *args, use_graph=False)
        launches[u8.shape[2]] = lib.t3d_launch_count() - n0
        _fused_from_plan(out)
    assert launches[512] == launches[384] - 3, launches


def _slab_step(full, sides, caps_of, world):
    """t3d_reconstruct_slab + t3d_slab_stitch_faces with all ranks emulated on one GPU (device copies stand in for the
    NCCL halo exchange and the all-gather of the result blocks).  Returns (plans, gathered host result blocks, outputs)."""
    from tomography_3d_reconstructor_b200 import sharded
    Z, H, W = (int(s) for s in full.shape)
    ranges = [sharded.slab_range(Z, r, world) for r in range(world)]
    plans = [sharded.FusedSlabPlan(b - a, H, W, Z, a, THRESHOLD, sides, *PHYS, 3, True, caps_of(r), full.device, r, world)
             for r, (a, b) in enumerate(ranges)]
    for pl, (a, b) in zip(plans, ranges):
        pl.pack(full[a:b].contiguous())
    for r, s in enumerate(plans):
        if s.hl:
            lo = plans[r - 1]
            s.ext[:s.hl] = lo.ext[lo.hl + lo.n - s.hl:lo.hl + lo.n]
        if s.hh:
            hi = plans[r + 1]
            s.ext[s.hl + s.n:] = hi.ext[hi.hl:hi.hl + s.hh]
    for pl in plans:
        pl.compute()
    gathered = torch.stack([pl.res for pl in plans])
    for pl in plans:
        pl.gathered.copy_(gathered)
        pl.stitch()
    h = gathered.cpu().numpy()
    return plans, h, [sharded.assemble(pl, h) for pl in plans]


def _slab_planes(pl):
    """Planes of the padded sign volume one slab step marches (Zs of its canonicalisation)."""
    from tomography_3d_reconstructor_b200 import sharded
    return min(sharded.SURF_HALO, pl.hl) + pl.n + min(sharded.SURF_HALO, pl.hh) + 2


SLAB_SHAPE = (48, 41, 512)


@pytest.mark.parametrize("zsort", [1, 8])
@pytest.mark.parametrize("world", [2, 3])
def test_morph4_slab_step_stitches_to_the_staged_mesh_and_the_oracle(eng, oracle, world, zsort):
    """Fused slab step at W = 512: pre-filled pack and k_morph4 with z0 > 0 on halo planes, both layer-sort variants
    (forced through cap_z); the stitched mesh must equal the staged path (four-launch chain) and the oracle bit for bit."""
    from tomography_3d_reconstructor_b200 import pipeline
    Z, H, W = SLAB_SHAPE
    sides = _sides(Z)
    u8 = _volume("blobs_s2", SLAB_SHAPE)
    ref = _reference("blobs_s2", SLAB_SHAPE)
    full = torch.from_numpy(u8).cuda()
    staged = pipeline.reconstruct(full, THRESHOLD, sides, *PHYS)
    rm = staged["mesh"]
    whole = pipeline._caps_from(rm.n_active, *rm.n_raw, rm.n_z, rm.n_raw[0])     # generous: the whole mesh per rank
    big_z = 4096 * (Z + 2)
    plans, h, _ = _slab_step(full, sides, lambda r: whole[:3] + (max(whole[3], big_z),) + whole[4:], world)
    n_z = [int(h[r, pipeline.R_NZ]) for r in range(world)]
    zs = [_slab_planes(pl) for pl in plans]
    if zsort == 8:
        caps = [whole[:3] + (max(whole[3], big_z),) + whole[4:] for _ in range(world)]
    else:
        caps = [whole[:3] + (pipeline._grow(n_z[r]),) + whole[4:] for r in range(world)]
    assert all(zsort_batched(c[3], s) == (zsort == 8) for c, s in zip(caps, zs)), (caps, zs)
    plans, h, outs = _slab_step(full, sides, lambda r: caps[r], world)
    assert all(pl.pre_active for pl in plans) and all(pl.n >= 16 for pl in plans)
    assert all(morph4_eligible(pl.hl + pl.n + pl.hh, H, W) for pl in plans)
    assert not h[:, pipeline.R_OVERFLOW].any() and not h[:, pipeline.R_UNVERIFIED].any()
    assert all(o["stitch_consistent"] for o in outs)
    v = torch.cat([o["verts"] for o in outs]).cpu().numpy()
    f = torch.cat([o["faces"] for o in outs]).cpu().numpy()
    rv, rf = rm.verts.cpu().numpy(), rm.faces.cpu().numpy()
    assert np.array_equal(v.view(np.uint32), rv.view(np.uint32)) and np.array_equal(f, rf)
    assert np.array_equal(v.view(np.uint32), ref["vertices"].view(np.uint32)) and np.array_equal(f, ref["faces"])
    o = outs[-1]
    assert o["voxel_volume_mm3"] == ref["voxel_volume"] == staged["voxel_volume_mm3"]
    assert o["processed_voxel_volume_mm3"] == ref["processed_volume"] == staged["processed_voxel_volume_mm3"]
    assert o["total_vertices"] == len(rv) and o["total_faces"] == len(rf)


# ----------------------------------------------------------------------------------------------------------------
# 2. bulk SDF passes against scipy
# ----------------------------------------------------------------------------------------------------------------
SDF_SHAPES = [
    (8, 70, 1024),      # y bulk, 5 chunks per line: the 3-stage ring wraps inside a tile
    (20, 60, 128),      # y bulk at the narrowest bulk width; z bulk, 2 chunks
    (300, 5, 1024),     # y pass: more lines than one resident wave -> several tiles per CTA; z: 19 chunks per line
    (5, 300, 1024),     # z pass: several tiles per CTA; y: 19 chunks per line
    (20, 9, 200),       # z bulk with a partial last tile (H*W mod 128 = 8); y not bulk
    (16, 13, 136),      # z bulk with a partial last tile (H*W mod 128 = 104); y not bulk
    (33, 13, 100),      # neither pass bulk (H*W mod 8 = 4)
]
SAMPLINGS = [(1.0, 1.0, 1.0), (0.09375, 0.31, 0.28)]


def test_sdf_shapes_cover_bulk_and_plain_passes():
    modes = [sdf_bulk_passes(*s) for s in SDF_SHAPES]
    assert {m[0] for m in modes} == {True, False} and {m[1] for m in modes} == {True, False}
    assert sdf_bulk_passes(8, 70, 1024) == (True, True) and sdf_bulk_passes(33, 13, 100) == (False, False)
    assert sdf_bulk_passes(20, 9, 200) == (False, True) and sdf_bulk_passes(16, 13, 136) == (False, True)
    for Z, H, W in SDF_SHAPES:
        if sdf_bulk_passes(Z, H, W)[1] and (H * W) % 128:
            assert 8 <= (H * W) % 128 <= 120
    # more lines than 148 SMs x 16 CTAs x 128 lines: several tiles per persistent CTA on any occupancy
    assert 300 * 1024 > 148 * MAX_CTAS_PER_SM * 128


def _sdf_volume(shape, kind):
    Z, H, W = shape
    rng = np.random.default_rng(Z * 7 + H * 3 + W + len(kind))
    if kind == "blobs":
        vol = random_blobs(rng, shape, 0.45, 1.5)
    elif kind == "noise":
        vol = rng.random(shape) < 0.5
    else:
        vol = rng.random(shape) < 0.02
    vol[Z // 3] = True                     # an all-ones plane and an all-zeros plane inside a mixed volume
    vol[(2 * Z) // 3 if Z > 2 else Z - 1] = False
    vol[:, H // 2, : W // 2] = True        # a half plane of ones across all z (z lines without any zero)
    return vol


@pytest.mark.parametrize("shape", SDF_SHAPES, ids=lambda s: "x".join(map(str, s)))
@pytest.mark.parametrize("sampling", SAMPLINGS, ids=["unit", "aniso"])
@pytest.mark.parametrize("kind", ["blobs", "noise", "sparse"])
def test_bulk_sdf_passes_match_scipy(eng, oracle, shape, sampling, kind):
    """t3d_sdf on shapes that run the bulk tile ring (wrapping rings, several tiles per CTA, partial last tiles) and on
    shapes that do not, against scipy's distance_transform_edt and against the two one-sided transforms."""
    from tomography_3d_reconstructor_b200 import edt
    Z, H, W = shape
    if shape in ((300, 5, 1024),):
        assert Z * W > _sm_count() * MAX_CTAS_PER_SM * 128
    if shape in ((5, 300, 1024),):
        assert H * W > _sm_count() * MAX_CTAS_PER_SM * 128
    vol = _sdf_volume(shape, kind)
    dv = dev_volume(eng, vol)
    got = edt.signed_distance(dv, sampling).cpu().numpy()
    two = edt.signed_distance_two_transforms(dv, sampling).cpu().numpy()
    ref = oracle.signed_distance(vol, sampling)
    if sampling == (1.0, 1.0, 1.0):
        assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
        assert np.array_equal(got.view(np.uint32), two.view(np.uint32))
    else:
        fin = np.isfinite(ref)
        assert np.array_equal(np.isfinite(got), fin)
        assert np.allclose(got[fin], ref[fin], rtol=1e-6, atol=0) and np.allclose(got[fin], two[fin], rtol=1e-6, atol=0)
        assert np.array_equal(got[~fin], ref[~fin])


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_bulk_sdf_matches_scipy(eng, oracle, world):
    """z-slab sharded signed distance at W = 256 (slab x/y pass and y-slab z pass both in bulk mode), all ranks emulated
    on one GPU, against scipy (the single-device transform runs the same bulk passes, so it is no independent check)."""
    from tomography_3d_reconstructor_b200 import edt, sharded
    Z, H, W = shape = (30, 37, 256)
    vol = _sdf_volume(shape, "blobs")
    dv = dev_volume(eng, vol)
    ranges = [sharded.slab_range(Z, r, world) for r in range(world)]
    for r, (a, b) in enumerate(ranges):
        a_h, b_h = edt.transpose_plan(Z, H, W, r, world)[1][r]
        assert sdf_bulk_ok(0, 0, (b - a) * W, W, H * W, W)                            # slab x/y pass
        assert sdf_bulk_ok(0, 0, (b_h - a_h) * W, (b_h - a_h) * W, 0, (b_h - a_h) * W)  # y-slab z pass
    ts = [edt.SlabTransform(dv.bits[a:b].contiguous(), Z, a, H, W, (1.0, 1.0, 1.0), r, world) for r, (a, b) in enumerate(ranges)]
    sends = [t.sdf_xy_pass() for t in ts]
    for c in range(2):
        _emulated_all_to_all([s[c] for s in sends], [t.send_sizes for t in ts], [t.cols[c] for t in ts], [t.recv_sizes for t in ts])
    for t in ts:
        t.sdf_z_pass()
    _emulated_all_to_all([t.dist_cols for t in ts], [t.recv_sizes for t in ts], [t.back for t in ts], [t.send_sizes for t in ts])
    out = torch.cat([t.result() for t in ts]).cpu().numpy()
    assert np.array_equal(out.view(np.uint32), oracle.signed_distance(vol).view(np.uint32))


# ----------------------------------------------------------------------------------------------------------------
# 3. k_zsort_layers<8> against the oracle
# ----------------------------------------------------------------------------------------------------------------
ZSORT_CASES = [("blobs_s2", SLAB_SHAPE), ("ellipsoid", (40, 300, 400)), ("plate", (24, 64, 500))]


@pytest.mark.parametrize("kind,shape", ZSORT_CASES, ids=[k for k, _ in ZSORT_CASES])
def test_layer_sort_variants_match_the_oracle(eng, oracle, kind, shape):
    """The same volume through the fused step with the per-layer z sort k_zsort_layers<1> (learned cap_z) and <8> (cap_z
    raised to 4096 planes); both bit-identical to each other and to the oracle, with a verified order (no fallback)."""
    from tomography_3d_reconstructor_b200 import pipeline
    Z, H, W = shape
    u8 = _volume(kind, shape)
    ref = _reference(kind, shape)
    masks = torch.from_numpy(u8).cuda()
    args = (THRESHOLD, _sides(Z), *PHYS)
    _clear_plans()
    pipeline.reconstruct_fused(masks, *args, use_graph=False)          # staged: learns the sizes
    (key, learned), = pipeline._hints.items()
    Zs = Z + 2
    assert not zsort_batched(learned[3], Zs), "the learned capacity already selects <8>: <1> cannot be reached"
    meshes = {}
    for variant in (1, 8):
        pipeline._plans.clear()
        cap_z = learned[3] if variant == 1 else max(learned[3], 4096 * Zs)
        pipeline._hints[key] = learned[:3] + (cap_z,) + learned[4:]
        for rep in range(2):       # (the first run may provision the clamp-group sort and re-run)
            out = pipeline.reconstruct_fused(masks, *args, use_graph=False)
            plan = _fused_from_plan(out)
            assert plan.caps[3] == cap_z and zsort_batched(plan.caps[3], Zs) == (variant == 8)
            _assert_matches_oracle(out, ref, plan, Z)
        v, f = out["mesh"].verts.cpu().numpy(), out["mesh"].faces.cpu().numpy()
        assert int(plan.res_np[pipeline.R_NZ]) > 1000
        meshes[variant] = (v.view(np.uint32).copy(), f.copy())
    assert np.array_equal(meshes[1][0], meshes[8][0]) and np.array_equal(meshes[1][1], meshes[8][1])
