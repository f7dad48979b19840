#!/usr/bin/env python3
"""bench.py -- headline benchmark: Gvoxels/s, mask stack -> stitched mesh + volumes (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape Z,H,W] [--dump-outputs DIR]

One "step" = one pass of the whole hot path over one synthetic ellipsoid mask stack (SURVEY.md 8d):
uint8 masks -> threshold+bit-pack -> close ends -> opening/closing -> Gaussian field sign -> two-pass marching
cubes -> canonical mesh -> mesh volume/area + voxel-count volumes.  N=1 workload = BASELINE.json configs[1]
(512 slices of 1024x1024).  N>1: the stack grows with N (512*N slices), z-slab sharded with NCCL halo exchange and
mesh stitching (weak scaling).  `value` has inputs resident in HBM; `e2e` goes through the reference-facing classes
with host buffers (H2D + D2H inside the timed region).  `--impl reference` times the CPU oracle (the restated
reference pipeline; the unmodified reference cannot run without scikit-image) on a bounded z-slab sample.
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Gvoxels/s mask-stack->mesh+volume"
PHYS = dict(x_length_mm=143.1, y_length_mm=95.03, total_depth_mm=6.0)  # config.py:12-14
THRESHOLD = 200                                                        # config.py:27


def side_counts(Z):
    s0 = Z // 8
    return (s0, Z - 2 * s0, s0)


# ----------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle (CPU restatement of the reference pipeline) on a bounded z-slab sample
# ----------------------------------------------------------------------------------------------------------------
def _cpu_sample_job(args):
    Z, H, W, z0, z1, sides, kind = args
    from oracle import cpu_ref
    u8 = cpu_ref.ellipsoid_phantom_u8(Z, H, W, z0, z1)
    sides = sides or side_counts(z1 - z0)
    t0 = time.perf_counter()
    if kind == "sdf":       # additive stage: smoothing -> scipy's exact EDT (both polarities) -> marching cubes at level 0
        masks = [u8[z] >= THRESHOLD for z in range(u8.shape[0])]
        sm = cpu_ref.smooth_voxel_data(cpu_ref.create_voxel_data(masks, True), 3, True)
        sdf = cpu_ref.signed_distance(sm, (PHYS["total_depth_mm"] / Z, PHYS["y_length_mm"] / H, PHYS["x_length_mm"] / W))
        cpu_ref.marching_cubes(sdf, 0.0)
    else:
        cpu_ref.reference_pipeline(u8, THRESHOLD, sides, PHYS["total_depth_mm"], PHYS["x_length_mm"], PHYS["y_length_mm"])
    return time.perf_counter() - t0, (z1 - z0) * H * W


def cpu_sample(Z, H, W, n_slices, workers, sides=None, kind="occupancy"):
    """Run the oracle on `workers` disjoint central z-slabs of n_slices each, in parallel processes (sides given: every
    worker runs the WHOLE stack, i.e. `workers` replicas).  Returns (seconds, voxels, slices per worker)."""
    import multiprocessing as mp
    if sides is not None:
        n_slices = Z
        jobs = [(Z, H, W, 0, Z, tuple(sides), kind) for _ in range(workers)]
    else:
        n_slices = max(4, min(n_slices, Z // max(1, workers)))
        zc = Z // 2 - (n_slices * workers) // 2
        jobs = [(Z, H, W, zc + k * n_slices, zc + (k + 1) * n_slices, None, kind) for k in range(workers)]
    t0 = time.perf_counter()
    if workers == 1:
        res = [_cpu_sample_job(jobs[0])]
    else:
        with mp.get_context("spawn").Pool(workers) as pool:
            res = pool.map(_cpu_sample_job, jobs)
    wall = time.perf_counter() - t0
    if workers > 1:
        wall = max(r[0] for r in res)  # exclude process start-up
    return wall, sum(r[1] for r in res), n_slices


def run_reference(args, Z, H, W, cfg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cpu_ref
    cpu_ref.build()
    cores = os.cpu_count() or 1
    workers = max(1, min(cores, 16))
    path = cfg["path"]
    kind = "sdf" if path == "sdf" else "occupancy"
    budget_per_step = 150.0 / max(1, args.steps + args.warmup)
    whole = path == "batch" or args.config == "C0"       # volumes small enough to run whole: one per worker
    sides = (cfg.get("sides") or side_counts(Z)) if whole else None
    # measured oracle speed is ~2.5 Mvox/s per core (scipy.ndimage is single-threaded); the EDT is ~4x slower
    n_slices = int(max(4, min(32, budget_per_step * (0.6e6 if kind == "sdf" else 2.5e6) / (H * W))))
    for _ in range(args.warmup):
        cpu_sample(Z, H, W, n_slices, workers, sides, kind)
    secs, vox = 0.0, 0
    for _ in range(args.steps):
        s, v, n_slices = cpu_sample(Z, H, W, n_slices, workers, sides, kind)
        secs += s
        vox += v
    value = vox / secs / 1e9
    if whole:
        sample = "%d whole %dx%dx%d stacks per step (one per worker process)" % (workers, Z, H, W)
    else:
        sample = "%d disjoint central z-slabs of %d slices x %dx%d per step (one per worker process)" % (workers, n_slices, H, W)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "Gvoxels/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bool/f64 (numpy/scipy)",
        "data": "synthetic",
        "config": {"workload": "%s, ellipsoid stack %dx%dx%d (bounded sample per step)" % (cfg["name"], Z, H, W), "config": args.config,
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Gvoxels/s", "cores": workers, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Gvoxels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append((time.perf_counter(), ln.strip()))

    def n_rows(self):
        return len(self.rows)

    def window(self, t0, t1):
        """Timed region [t0, t1] (perf_counter); samples inside it are counted apart in summary()."""
        self.t0, self.t1 = t0, t1

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons, inside = [], [], set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            if self.t0 is not None and self.t0 <= ts <= self.t1 + 0.1:
                inside += 1
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm),
                "samples_in_timed_region": inside,
                "note": "sampled every 100 ms while the same step runs back to back (load phase before + timed region + load phase "
                        "after): the timed region itself can be shorter than one sampling period"}


def make_phantom_u8(Z_total, H, W, z0, z1, device):
    """Analytic ellipsoid of SURVEY.md 8d, slices [z0, z1) of a Z_total stack, uint8 0/255, built on the device."""
    import torch
    cz, cy, cx = Z_total / 2 - 0.3, H / 2 + 0.2, W / 2 - 0.1
    rz, ry, rx = 0.42 * Z_total, 0.33 * H, 0.45 * W
    out = torch.empty((z1 - z0, H, W), dtype=torch.uint8, device=device)
    y = ((torch.arange(H, dtype=torch.float64, device=device) - cy) / ry) ** 2
    x = ((torch.arange(W, dtype=torch.float64, device=device) - cx) / rx) ** 2
    yx = y[:, None] + x[None, :]
    for a in range(z0, z1, 16):
        b = min(z1, a + 16)
        z = ((torch.arange(a, b, dtype=torch.float64, device=device) - cz) / rz) ** 2
        out[a - z0:b - z0] = ((z[:, None, None] + yx[None]) <= 1.0).to(torch.uint8) * 255
    return out


NCU_PACK_TRAFFIC_BYTES = 567000000   # k_pack_gap at C1: 552.3 MB read + 14.7 MB written (profiles/r02_ncu_full_pack_gap_and_staged_path_c1.txt)

STAGE_BYTES = {  # algorithmic bytes per voxel of each volume-sized stage (DESIGN.md section 4)
    "pack_close": 1.0 + 0.125 + 0.25, "smooth": 4 * 0.25, "field_sign": 0.25, "mc_flags": 0.125 + 1.0 / 256,
}

# BASELINE.json configs -> (per-GPU shape, path).  The stack grows with the number of GPUs (weak scaling): C3 / C4 are the
# full 2048^3 / 4096^3 stacks at N = 8 and one GPU's z-slab of them at N = 1.
CONFIGS = {
    "C0": dict(shape=(104, 512, 512), sides=(20, 64, 20), path="occupancy", replicas=True,
               name="C0 (BASELINE configs[0]): 512x512 masks, Section_0/1/2 = 20+64+20 slices"),
    "C1": dict(shape=(512, 1024, 1024), path="occupancy", name="C1 (BASELINE configs[1])"),
    "C2": dict(shape=(256, 256, 256), path="batch", count=256,
               name="C2 (BASELINE configs[2]): batch of 256 independent 256^3 phantoms, round robin over the GPUs"),
    "C3": dict(shape=(256, 2048, 2048), path="sdf",
               name="C3 (BASELINE configs[3]): 2048x2048 slices, exact EDT/SDF + marching cubes on the distance field, "
                    "256 slices per GPU (the full 2048^3 stack at 8 GPUs)"),
    "C4": dict(shape=(512, 4096, 4096), path="occupancy",
               name="C4 (BASELINE configs[4]): 4096x4096 slices, 512 per GPU (the full 4096^3 stack at 8 GPUs)"),
}


def mesh_digest(v, f):
    """sha256 over the float32 vertex bits and the int64 faces of a device mesh (downloaded in chunks)."""
    import hashlib
    h = hashlib.sha256()
    for t in (v, f):
        t = t.contiguous()
        flat = t.view(-1)
        for a in range(0, flat.numel(), 1 << 24):
            h.update(flat[a:a + (1 << 24)].cpu().numpy().tobytes())
    return h.hexdigest()[:16]


def mesh_topology(v, f):
    """(closed oriented 2-manifold?, Euler characteristic) of a device mesh: every directed edge once and its twin present."""
    import torch
    V = int(v.shape[0])
    e = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    key = e[:, 0] * (V + 1) + e[:, 1]
    rev = e[:, 1] * (V + 1) + e[:, 0]
    sk = torch.sort(key)[0]
    closed = bool((sk[1:] != sk[:-1]).all()) and bool(torch.equal(sk, torch.sort(rev)[0]))
    return closed, V - int(key.numel()) // 2 + int(f.shape[0])


DUMP_BYTES = 60 * 10 ** 6      # --dump-outputs: under 64 MB with the .npy headers
BATCH_FIELDS = ("voxel_volume_mm3", "processed_voxel_volume_mm3", "mesh_volume_mm3", "surface_area_mm2", "active_voxels",
                "n_vertices", "n_faces", "n_ambiguous")


def step_outputs(res, path):
    """What a caller of the timed path receives from one step: name -> tensor / array / scalar."""
    import torch
    if path == "batch":      # {volume index: that volume's scalars}
        items = sorted(res)
        out = {"volume_index": np.array(items)}
        out.update({k: np.array([res[i][k] for i in items]) for k in BATCH_FIELDS})
        out["bbox_index"] = np.array([res[i]["bbox_index"] or (np.nan,) * 6 for i in items])   # (an empty volume has none)
        return out
    out = {"vertices": res["mesh"].verts, "faces": res["mesh"].faces}
    for k, v in res.items():
        if k in ("mesh", "verts", "faces"):          # (a sharded step also returns the mesh arrays under these names)
            continue
        if isinstance(v, (torch.Tensor, np.ndarray, bool, int, float)) or (k == "bbox_index" and v is not None):
            out[k] = v
    return out


def dump_outputs(outputs, dirpath, budget):
    """Write every output as <name>.npy, float32 kept and everything else as float64 (integers are exact below 2**53),
    `budget` bytes in all.  An array larger than its share is replaced by a fixed seeded sample of its rows (elements of
    a 3-D field), the sorted row indices written beside it as <name>_rows.npy.  Copies to the host before it returns."""
    import torch
    os.makedirs(dirpath, exist_ok=True)
    items = []
    for name, v in outputs.items():
        t = v if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v))
        t = t.reshape(t.shape[0], -1) if t.dim() == 2 else t.reshape(-1) if t.dim() > 2 else t
        items.append((t.numel() * (4 if t.dtype == torch.float32 else 8), name, t))
    items.sort(key=lambda x: x[0])
    left = budget
    for k, (nbytes, name, t) in enumerate(items):
        share = left // (len(items) - k)
        if nbytes > share:
            row_bytes = nbytes // t.shape[0] + 8
            rows = np.unique(np.random.default_rng(0).integers(0, t.shape[0], share // row_bytes))
            np.save(os.path.join(dirpath, name + "_rows.npy"), rows.astype(np.float64))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
            nbytes = t.numel() * (4 if t.dtype == torch.float32 else 8) + 8 * len(rows)
        a = t.cpu().numpy()
        np.save(os.path.join(dirpath, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))
        left -= nbytes


def sharded_check(world, rank, dev, H=512, W=512, per_rank=128):
    """N > 1: the stitched mesh of a (per_rank*N, H, W) stack sharded over the N ranks against rank 0's own single-GPU run
    of the same stack: same bits (sha256 of vertices + faces), closed 2-manifold, Euler characteristic 2, consistent
    ghost/lead stitching, same volumes.  Asserted, and reported in the bench line."""
    import torch
    import torch.distributed as dist
    from tomography_3d_reconstructor_b200 import pipeline, sharded
    Zc = per_rank * world
    sides = side_counts(Zc)
    phys = (PHYS["total_depth_mm"], PHYS["x_length_mm"], PHYS["y_length_mm"])
    z0, z1 = sharded.slab_range(Zc, rank, world)
    masks = make_phantom_u8(Zc, H, W, z0, z1, dev)
    for _ in range(3):     # staged (learns the sizes), fused, fused + graph
        out = sharded.reconstruct_fused(masks, Zc, z0, THRESHOLD, sides, *phys, use_graph=True)
    gm = sharded.gather_mesh(out, 0)
    rep = None
    if rank == 0:
        v, f = gm
        full = make_phantom_u8(Zc, H, W, 0, Zc, dev)
        for _ in range(2):
            ref = pipeline.reconstruct_fused(full, THRESHOLD, sides, *phys)
        rv, rf = ref["mesh"].verts, ref["mesh"].faces
        closed, euler = mesh_topology(v, f)
        rep = {"shape": [Zc, H, W], "ranks": world, "vertices": int(v.shape[0]), "faces": int(f.shape[0]),
               "mesh_sha256_16": mesh_digest(v, f), "single_gpu_sha256_16": mesh_digest(rv, rf),
               "stitch_consistent": bool(out["stitch_consistent"]), "closed_manifold": closed, "euler": euler,
               "voxel_volume_equal": out["voxel_volume_mm3"] == ref["voxel_volume_mm3"],
               "processed_volume_equal": out["processed_voxel_volume_mm3"] == ref["processed_voxel_volume_mm3"],
               "bbox_equal": out["bbox_index"] == ref["bbox_index"],
               "mesh_volume_rel_diff": abs(out["mesh_volume_mm3"] - ref["mesh_volume_mm3"]) / ref["mesh_volume_mm3"]}
        rep["ok"] = bool(rep["mesh_sha256_16"] == rep["single_gpu_sha256_16"] and rep["stitch_consistent"] and closed and euler == 2
                         and rep["voxel_volume_equal"] and rep["processed_volume_equal"] and rep["bbox_equal"]
                         and rep["mesh_volume_rel_diff"] <= 1e-9)
        del full, ref
    sharded._slab_plans.clear()
    pipeline._plans.clear()
    del masks, out, gm
    torch.cuda.empty_cache()
    flag = torch.tensor([0 if (rep is None or rep["ok"]) else 1], device=dev)
    dist.all_reduce(flag)
    if int(flag.item()):
        raise AssertionError("sharded mesh differs from the single-GPU mesh: %r" % (rep,))
    return rep


def run_ours(args, Z, H, W, cfg):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL's own logging is left exactly as the caller set it (NCCL_DEBUG / NCCL_DEBUG_FILE); the JSON line is the LAST
        # line this program prints to stdout
        dist.init_process_group("nccl", device_id=dev)
    from tomography_3d_reconstructor_b200 import _lib, engine, pipeline
    lib = _lib.load()
    path = cfg["path"]
    replicas = bool(cfg.get("replicas")) or path == "batch"
    phys = (PHYS["total_depth_mm"], PHYS["x_length_mm"], PHYS["y_length_mm"])

    if replicas:
        Zg, z0, z1 = Z, 0, Z                 # every rank holds whole volumes: no collective on the data path
    else:
        Zg = Z * world                       # weak scaling: the stack grows with the number of GPUs
        if world > 1:
            from tomography_3d_reconstructor_b200 import sharded
            z0, z1 = sharded.slab_range(Zg, rank, world)
        else:
            z0, z1 = 0, Zg
    sides = cfg.get("sides") or side_counts(Zg)
    sharded_run = world > 1 and not replicas
    if sharded_run:
        from tomography_3d_reconstructor_b200 import sharded

    if path == "batch":
        from tomography_3d_reconstructor_b200 import batch
        count = int(cfg["count"])
        radii, centres = batch.phantom_params(count, Z)
        mine = batch.my_items(count, rank, world)
        stacks = {i: batch.phantom_u8(Z, radii[i], centres[i], dev) for i in mine}
        masks = None
        voxels = count * Z * H * W
        per_gpu_vox = len(mine) * Z * H * W
    else:
        masks = make_phantom_u8(Zg, H, W, z0, z1, dev)
        voxels = Zg * H * W * (world if replicas else 1)
        per_gpu_vox = (z1 - z0) * H * W

    def step(mark=None):
        if path == "batch":
            return batch.reconstruct_volumes(stacks, THRESHOLD, sides, *phys)
        if path == "sdf":
            if sharded_run:
                return sharded.reconstruct_sdf(masks, Zg, z0, THRESHOLD, sides, *phys)
            return pipeline.reconstruct_sdf(masks, THRESHOLD, sides, *phys)
        if sharded_run:
            if mark is not None or args.staged:
                return sharded.reconstruct(masks, Zg, z0, THRESHOLD, sides, *phys, mark=mark)
            # fused: pack -> NCCL halo exchange -> one t3d_reconstruct_slab enqueue -> all-gather -> stitch, one sync
            return sharded.reconstruct_fused(masks, Zg, z0, THRESHOLD, sides, *phys, use_graph=not args.no_graph)
        if mark is not None or args.staged:   # staged path: one library call per stage (per-stage event timing)
            return pipeline.reconstruct(masks, THRESHOLD, sides, *phys, mark=mark)
        # fused path: the whole step is one t3d_reconstruct enqueue replayed from a CUDA graph + one D2H copy
        return pipeline.reconstruct_fused(masks, THRESHOLD, sides, *phys, use_graph=not args.no_graph)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_ranks_agree(flag):
        """True on every rank iff rank 0 says so (steps are collective when sharded: every rank must stop together)."""
        if world == 1:
            return flag
        t = torch.tensor([1 if flag else 0], device=dev)
        dist.broadcast(t, 0)
        return bool(t.item())

    for _ in range(max(3, args.warmup)):
        res = step()
    barrier()
    partition = None
    if sharded_run and path == "occupancy" and not args.no_balance:
        # Equal slice counts are equal voxel work but unequal surface work (polar slabs carry less mesh than equatorial ones),
        # and the step ends with a collective: re-cut the slabs by estimated cost, learned from the equal-split step above
        hist = torch.from_numpy(sharded.vertices_per_slice(res, Zg)).to(dev)
        dist.all_reduce(hist)
        # (the volume passes of a slice cost about as much as ~2900 mesh vertices at 1024x1024, in proportion to the slice area)
        # cost of a slice in units of one surface vertex.  Kernel times alone say ~1950 (volume kernels ~0.38 us per 1024 x 1024
        # slice, mesh kernels ~0.19 us per 1000 vertices), but the end ranks also fill the holes of an end slice and sort the
        # large polar layers: measured at N = 8, 2900 beats 1950 (C1 0.750 against 0.783 ms per step, 4096^3 5.32 against 5.51 ms;
        # profiles/r02_balance_constant_n8.txt).  T3D_BALANCE_SLICE_COST overrides it.
        slice_units = float(os.environ.get("T3D_BALANCE_SLICE_COST", "2900")) * (H * W) / (1024.0 * 1024.0)
        partition = sharded.balanced_ranges(sharded.slice_cost(hist.cpu().numpy(), slice_units), world,
                                            sharded.HALO)
        sharded.set_partition(Zg, world, partition)
        z0, z1 = partition[rank]
        del masks
        torch.cuda.empty_cache()
        masks = make_phantom_u8(Zg, H, W, z0, z1, dev)
        per_gpu_vox = (z1 - z0) * H * W
        for _ in range(max(3, args.warmup)):
            res = step()
        barrier()
    # kernels of this library per step: counted on one eager (non-graph) step, a graph replay launches the same ones
    lc0 = lib.t3d_launch_count()
    if path == "occupancy" and not args.staged:
        if sharded_run:
            sharded.reconstruct_fused(masks, Zg, z0, THRESHOLD, sides, *phys, use_graph=False)
        else:
            pipeline.reconstruct_fused(masks, THRESHOLD, sides, *phys, use_graph=False)
    elif path == "batch":
        # every volume of the batch is one t3d_reconstruct enqueue replayed from its slot's graph: count one eager enqueue of one
        # volume of this shape (after a staged call that learns its capacities) and multiply
        one = next(iter(stacks.values()))
        pipeline.reconstruct_fused(one, THRESHOLD, sides, *phys, use_graph=False)
        lc0 = lib.t3d_launch_count()
        pipeline.reconstruct_fused(one, THRESHOLD, sides, *phys, use_graph=False)
        lc0 -= (lib.t3d_launch_count() - lc0) * (len(stacks) - 1)
    else:
        step()
    launches_per_step = lib.t3d_launch_count() - lc0
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        # load phase: the same step back to back until the sampler has delivered a few rows (a C1 step is ~1 ms, the
        # sampling period 100 ms), then the timed region, then a short load phase again so that samples bracket it
        t_load = time.perf_counter()
        while not all_ranks_agree(clocks.n_rows() >= 3 or time.perf_counter() - t_load > 4.0):
            for _ in range(10 if path == "occupancy" else 1):
                step()
        barrier()
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(args.steps):
            res = step()
        ev1.record()
        barrier()
        t1 = time.perf_counter()
        clocks.window(t0, t1)
        if args.dump_outputs:
            # before any further step: the mesh of a fused step lives in its plan's buffers, which the next step overwrites
            dump_outputs(step_outputs(res, path), args.dump_outputs if world == 1 else
                         os.path.join(args.dump_outputs, "rank%d" % rank), DUMP_BYTES // world)
        n_before = clocks.n_rows()
        t_load = time.perf_counter()
        while not all_ranks_agree(clocks.n_rows() >= n_before + 2 or time.perf_counter() - t_load > 1.0):
            for _ in range(10 if path == "occupancy" else 1):
                step()
        barrier()
    ms = ev0.elapsed_time(ev1)
    launches = launches_per_step
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = voxels * args.steps / (ms * 1e-3) / 1e9

    # ---- the kernel that moves the most bytes, timed alone on the launching stream: the mask decode / bit packing
    # streams the whole u8 stack (larger than L2) and writes the bit volume
    pack_ms = None
    if masks is not None:
        n_own = z1 - z0
        kbits = torch.empty((n_own, H, engine.words_per_row(W)), dtype=torch.int32, device=dev)
        kst = engine._stream()
        # the kernel the single-enqueue step streams the masks with: threshold + stack + z gap fill + per-slice counts
        # (k_pack_gap); stacks it does not take (W % 128 != 0, fewer than 3 slices) go through the plain pack kernel
        # (a sharded step runs the same kernel over the interior planes of its slab when the slab has >= 16 slices: t3d_slab_pack)
        pack_gap = n_own >= 3 and W % 128 == 0 and (not sharded_run or n_own >= 16)
        kstat = torch.empty(n_own + 3, dtype=torch.int64, device=dev)      # per-slice counts, then the 6 extrema (zeroed by one memset)
        kcnt, kbb = kstat[:n_own], kstat[n_own:].view(torch.int32)

        def pack_launch():
            if pack_gap:
                rc = lib.t3d_pack_gap(engine._p(masks), n_own, H, W, THRESHOLD, engine._p(kbits), engine._p(kcnt), engine._p(kbb), kst)
            else:
                rc = lib.t3d_pack_masks(engine._p(masks), n_own, H, W, THRESHOLD, engine._p(kbits), kst)
            if rc:
                raise RuntimeError("pack kernel failed: rc=%d" % rc)

        kstat.zero_()      # (t3d_pack_gap accumulates its counts / extrema: zeroed once, the timed launches are the kernel alone)
        for _ in range(3):
            pack_launch()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        K_REP = 20
        k0.record()
        for _ in range(K_REP):
            pack_launch()
        k1.record()
        torch.cuda.synchronize()
        pack_ms = k0.elapsed_time(k1) / K_REP
        del kbits

    # ---- per-stage device times (one instrumented step, events on the launching stream)
    marks = []

    def mark(name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        marks.append((name, e))

    stage_ms = {}
    if path == "occupancy":
        for _ in range(3):
            marks.clear()
            barrier()
            mark("start")
            step(mark)
            barrier()
            for (n0, e0), (n1, e1) in zip(marks[:-1], marks[1:]):
                stage_ms.setdefault(n1, []).append(e0.elapsed_time(e1))
        stage_ms = {k: float(np.min(v)) for k, v in stage_ms.items()}

    # ---- e2e through the reference-facing classes, host buffers in pinned memory
    e2e = e2e_classes = e2e_bits = None
    want_e2e = path == "occupancy" and not args.no_e2e
    if want_e2e and not sharded_run:
        from tomography_3d_reconstructor_b200 import VoxelProcessor, SurfaceExtractor, VolumeCalculator
        host_bool = torch.empty((Z, H, W), dtype=torch.bool, pin_memory=True)
        host_bool.copy_(masks >= THRESHOLD)          # image_loader.py:108 happens upstream of the hot path
        torch.cuda.synchronize()
        hb = host_bool.numpy()
        mask_list = [hb[z] for z in range(Z)]
        mm_x, mm_y = PHYS["x_length_mm"] / W, PHYS["y_length_mm"] / H

        def api_step():
            vp, se, vc = VoxelProcessor(), SurfaceExtractor(), VolumeCalculator()
            vox = vp.create_voxel_data(mask_list, True, *sides)
            depths = vp.calculate_slice_depths(PHYS["total_depth_mm"])
            sm = vp.smooth_voxel_data(vox, 3, True)
            processed = vc.calculate_voxel_volume_variable_depth(sm, mm_x, mm_y, depths)
            v, f = se.extract_manifold_surface(sm, depths, mm_y, mm_x, True, True, True)
            mv = se.calculate_mesh_volume(v, f)
            ar = se.calculate_surface_area(v, f)
            props = vc.analyze_object_properties(vox, processed, mv, ar, mm_x, mm_y, depths, PHYS["x_length_mm"],
                                                 PHYS["y_length_mm"], PHYS["total_depth_mm"])
            return vox, sm, v, f, props

        sink = io.StringIO()
        with contextlib.redirect_stdout(sink):
            for _ in range(4):      # (the first calls also populate torch's pinned-host allocator cache: 3 x 537 MB blocks)
                out = api_step()
            n_e2e = max(2, min(args.steps, 5))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                out = api_step()
            torch.cuda.synchronize()
            e2e_s = (time.perf_counter() - t0) / n_e2e
        vox, sm, v, f, props = out
        e2e_classes = {"value": voxels / world / e2e_s / 1e9, "unit": "Gvoxels/s", "h2d_bytes_per_step": int(hb.nbytes),
                       "d2h_bytes_per_step": int(vox.nbytes + sm.nbytes + v.nbytes + f.nbytes), "ms_per_step": 1e3 * e2e_s,
                       "steps": n_e2e, "api": "VoxelProcessor.create_voxel_data -> smooth_voxel_data -> "
                       "SurfaceExtractor.extract_manifold_surface -> calculate_mesh_volume/area -> "
                       "VolumeCalculator.analyze_object_properties (also returns both bool voxel grids to the host: 2 x 1 B/voxel)"}
        del out, vox, sm
        # the same work as one call: host masks in, host mesh + volumes out (what the reference arm computes)
        host_u8 = torch.empty((Z, H, W), dtype=torch.uint8, pin_memory=True)
        host_u8.copy_(masks)
        torch.cuda.synchronize()
        hu = host_u8.numpy()
        u8_list = [hu[z] for z in range(Z)]

        def host_step():
            return pipeline.reconstruct_host(u8_list, THRESHOLD, sides, *phys, use_graph=not args.no_graph)

        for _ in range(2):
            out = host_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            out = host_step()
        barrier()
        e2e_s = (time.perf_counter() - t0) / n_e2e
        if world > 1:
            tm = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            e2e_s = float(tm.item())
        e2e = {"value": voxels / e2e_s / 1e9, "unit": "Gvoxels/s", "h2d_bytes_per_step": int(hu.nbytes) * world,
               "d2h_bytes_per_step": int(out["vertices"].nbytes + out["faces"].nbytes + 8 * (32 + 2 * Z)) * world,
               "ms_per_step": 1e3 * e2e_s, "steps": n_e2e,
               "api": "pipeline.reconstruct_host: list of pinned host u8 masks -> H2D -> t3d_reconstruct -> D2H of the mesh "
               "(f32 vertices, int64 faces) and the result block (volumes, area, bbox, per-slice counts)"}
        assert np.array_equal(out["vertices"], v) and np.array_equal(out["faces"], f)
        # additive entry: the same masks already bit-packed on the host (1 bit per voxel over PCIe)
        if world == 1:
            from tomography_3d_reconstructor_b200 import sharded as _sh
            wpr = engine.words_per_row(W)
            host_bits = torch.empty((Z, H, wpr), dtype=torch.int32, pin_memory=True)
            packed = torch.empty((Z, H, wpr), dtype=torch.int32, device=dev)
            lib.t3d_pack_masks(engine._p(masks), Z, H, W, THRESHOLD, engine._p(packed), engine._stream())
            host_bits.copy_(packed)
            torch.cuda.synchronize()
            del packed
            hbits = host_bits.numpy().view(np.uint32)
            for _ in range(3):
                ob = _sh.reconstruct_host_bits(hbits, W, sides, *phys, use_graph=not args.no_graph)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n_e2e):
                ob = _sh.reconstruct_host_bits(hbits, W, sides, *phys, use_graph=not args.no_graph)
            torch.cuda.synchronize()
            eb_s = (time.perf_counter() - t0) / n_e2e
            assert np.array_equal(ob["vertices"], v) and np.array_equal(ob["faces"], f)
            e2e_bits = {"value": voxels / eb_s / 1e9, "unit": "Gvoxels/s", "h2d_bytes_per_step": int(hbits.nbytes),
                        "d2h_bytes_per_step": int(ob["vertices"].nbytes + ob["faces"].nbytes + 8 * (32 + 2 * Z)), "ms_per_step": 1e3 * eb_s,
                        "steps": n_e2e, "api": "sharded.reconstruct_host_bits: pinned host masks ALREADY bit-packed (1 bit per voxel) -> H2D -> "
                        "t3d_reconstruct_slab -> D2H of the mesh and the result block (additive input format; not the headline e2e)"}

    def teardown():
        if world > 1:
            # captured graphs hold NCCL work: release them before the communicator goes away
            if sharded_run:
                sharded._slab_plans.clear()
            import gc
            gc.collect()
            torch.cuda.synchronize()
            dist.barrier()
            dist.destroy_process_group()

    if want_e2e and sharded_run:
        # sharded e2e: every rank uploads its slab from pinned host memory and downloads its slab of the stitched mesh
        host_u8 = torch.empty((z1 - z0, H, W), dtype=torch.uint8, pin_memory=True)
        host_u8.copy_(masks)
        torch.cuda.synchronize()
        hnp = host_u8.numpy()

        def host_step():
            return sharded.reconstruct_host(hnp, Zg, z0, THRESHOLD, sides, *phys, use_graph=not args.no_graph)

        for _ in range(2):
            out = host_step()
        n_e2e = max(2, min(args.steps, 5))
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            out = host_step()
        barrier()
        e2e_s = (time.perf_counter() - t0) / n_e2e
        t = torch.tensor([e2e_s, float(hnp.nbytes), float(out["vertices_host"].nbytes + out["faces_host"].nbytes)],
                         dtype=torch.float64, device=dev)
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        e2e_s = float(tmax[0].item())
        e2e = {"value": voxels / e2e_s / 1e9, "unit": "Gvoxels/s", "h2d_bytes_per_step": int(t[1].item()),
               "d2h_bytes_per_step": int(t[2].item()), "ms_per_step": 1e3 * e2e_s, "steps": n_e2e,
               "api": "sharded.reconstruct_host: per-rank pinned host u8 slab -> H2D -> sharded step -> D2H of the rank's "
               "slab of the stitched mesh (bytes summed over ranks, time = max over ranks)"}

    # ---- N > 1: the stitched mesh against a single-GPU run of the same stack (asserted)
    check = None
    if sharded_run and path == "occupancy" and not args.no_check:
        del masks
        masks = None
        sharded._slab_plans.clear()
        torch.cuda.empty_cache()
        check = sharded_check(world, rank, dev)

    # mesh totals
    if path == "batch":
        tot = torch.tensor([sum(o["n_vertices"] for o in res.values()), sum(o["n_faces"] for o in res.values()),
                            sum(o["n_ambiguous"] for o in res.values())], dtype=torch.int64, device=dev)
        if world > 1:
            dist.all_reduce(tot)
        V, F, n_amb = (int(x) for x in tot.tolist())
        results = {"volumes": count, "first_volume_mesh_volume_mm3": float(res[mine[0]]["mesh_volume_mm3"]) if mine else None}
    else:
        mesh = res["mesh"]
        V = int(res.get("total_vertices", mesh.verts.shape[0]))
        F = int(res.get("total_faces", mesh.faces.shape[0]))
        n_amb = int(getattr(mesh, "n_ambiguous", 0))
        if replicas and world > 1:
            V, F = V * world, F * world
        results = {"voxel_volume_mm3": float(res["voxel_volume_mm3"]), "mesh_volume_mm3": float(res["mesh_volume_mm3"]),
                   "surface_area_mm2": float(res["surface_area_mm2"]), "active_voxels": int(res["active_voxels"])}
        if "stitch_consistent" in res:
            results["stitch_consistent"] = bool(res["stitch_consistent"])
            if not res["stitch_consistent"]:
                raise AssertionError("sharded step: ghost tail / lead mismatch between neighbouring ranks")

    if rank != 0:
        teardown()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    mesh_bytes = 12 * V + 12 * F
    # SURVEY.md 8(d): algorithmic bytes per voxel of the whole path + the mesh it writes
    per_voxel = 17.5 if path == "sdf" else 1.5
    bytes_alg = per_voxel * voxels + mesh_bytes
    step_gbs = bytes_alg * args.steps / (ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "scope": "whole step (every kernel of the path, SURVEY.md 8d)", "achieved": step_gbs,
                "peak": peak * world, "unit": "GB/s", "frac": step_gbs / (peak * world), "traffic": None,
                "peak_source": peak_src + (" x %d GPUs" % world if world > 1 else ""),
                "frac_of_nominal_8TBs": step_gbs / (8000.0 * world),     # SURVEY.md 8(d): also against the nominal 8 TB/s
                "algorithmic_bytes_per_step": bytes_alg,
                "algorithmic_bytes": "%.3g B/voxel x %d voxels + 12 B x (%d vertices + %d faces)" % (per_voxel, voxels, V, F)}
    if pack_ms is not None:
        dom_bytes = 1.125 * per_gpu_vox
        achieved = dom_bytes / (pack_ms * 1e-3) / 1e9
        roofline["dominant_kernel"] = {
            "kernel": ("k_pack_gap (t3d_pack_gap: threshold + stack + z gap fill + slice counts, the kernel of the step that streams "
                       "the u8 masks)" if pack_gap else "k_pack_flat (t3d_pack_masks)") + ": moves the most bytes of any kernel of the step",
            "achieved": achieved,
            "peak": peak, "unit": "GB/s", "frac": achieved / peak, "algorithmic_bytes_per_launch": dom_bytes,
            "us_per_launch": 1e3 * pack_ms, "launches_timed": 20, "share_of_step": pack_ms / (ms / args.steps),
            "traffic": NCU_PACK_TRAFFIC_BYTES if (Z, H, W) == (512, 1024, 1024) and pack_gap else None,
            "traffic_source": "profiles/r02_ncu_full_pack_gap_and_staged_path_c1.txt: ncu --set full of this kernel at C1, "
                              "dram__bytes_read.sum + dram__bytes_write.sum per launch (most of the 67 MB bit volume it writes "
                              "stays in the 126 MB L2)"}
    if stage_ms:
        roofline["stages"] = {k: {"GB/s": STAGE_BYTES[k] * per_gpu_vox / (stage_ms[k] * 1e-3) / 1e9,
                                  "frac": STAGE_BYTES[k] * per_gpu_vox / (stage_ms[k] * 1e-3) / 1e9 / peak}
                              for k in STAGE_BYTES if k in stage_ms}
    execution = {
        "batch": "batch.reconstruct_volumes: all volumes of a rank in one t3d_reconstruct_batch enqueue, replayed from a CUDA graph",
        "sdf": ("sharded.reconstruct_sdf: z-slab sharded, EDT z pass through an NCCL all-to-all transpose" if sharded_run
                else "pipeline.reconstruct_sdf"),
        "occupancy": ("z-slab sharded, staged launches" if sharded_run and args.staged else
                      "z-slab sharded: pack, NCCL halo exchange, one t3d_reconstruct_slab enqueue, result all-gather, "
                      "face stitching; one host sync per step" + ("" if args.no_graph else ", replayed from a CUDA graph (NCCL included)")
                      if sharded_run else "staged launches" if args.staged else
                      "one t3d_reconstruct enqueue per step" + ("" if args.no_graph else ", replayed from a CUDA graph")
                      + ("; %d independent replicas, no collective" % world if world > 1 else "")),
    }[path]
    line = {
        "metric": METRIC, "value": value, "unit": "Gvoxels/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8 -> bit-packed u32 (topology), f64 field taps -> f32 vertices", "data": "synthetic",
        "config": {"workload": "%s: %s analytic ellipsoid masks (u8 0/255), threshold 200, close ends + opening/closing + %s + volumes%s" %
                   (cfg["name"], "%d volumes of %dx%dx%d" % (cfg["count"], Z, H, W) if path == "batch" else
                    "%d slices of %dx%d" % (Zg, H, W),
                    "exact EDT/SDF + marching cubes at level 0" if path == "sdf" else "Gaussian(0.5) marching cubes",
                    "; z-slab sharded over %d GPUs" % world if sharded_run else ""),
                   "config": args.config, "shape": [Zg, H, W],
                   "partition": ("cost-balanced z-slabs (slices per GPU: %s), learned from one equal-split step" %
                                 [b - a for a, b in partition]) if partition else ("equal z-slabs" if sharded_run else None),
                   "l2": "inputs larger than L2: %.0f MB of u8 masks per GPU per step" % (per_gpu_vox / 1e6)
                   if per_gpu_vox > 130e6 else "inputs of one step (%.0f MB of u8 masks) fit the 126 MB L2" % (per_gpu_vox / 1e6),
                   "mesh": {"vertices": V, "faces": F, "n_ambiguous_cubes": n_amb},
                   "execution": execution},
        "clocks": clocks.summary(),
        "gpu_launches": int(launches),
        "stages_ms": stage_ms,
        "roofline": roofline,
        "results": results,
    }
    if check is not None:
        line["sharded_check"] = check
    if e2e is not None:
        line["e2e"] = e2e
    if e2e_classes is not None:
        line["e2e_classes"] = e2e_classes
    if e2e_bits is not None:
        line["e2e_bits"] = e2e_bits
    if world == 1 and not args.no_cpu and path == "occupancy":
        from oracle import cpu_ref
        cpu_ref.build()
        secs, vox_s, n_sl = cpu_sample(Z, H, W, 96, 1, sides if args.config == "C0" else None)
        line["cpu_baseline"] = {"value": vox_s / secs / 1e9, "unit": "Gvoxels/s", "cores": 1, "kind": "port",
                                "sample": "central z-slab of %d slices x %dx%d of the same phantom, oracle/cpu_ref.py "
                                "(scipy.ndimage is single-threaded), %.1f s" % (n_sl, H, W, secs)}
    teardown()
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C1", choices=sorted(CONFIGS), help="BASELINE.json configuration (C1 = configs[1], the headline)")
    ap.add_argument("--shape", default=None, help="Z,H,W per GPU (overrides the shape of --config; occupancy path)")
    ap.add_argument("--no-check", action="store_true", help="N>1: skip the stitched-mesh-vs-single-GPU check")
    ap.add_argument("--no-balance", action="store_true", help="N>1: equal slice counts per GPU instead of cost-balanced z-slabs")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--staged", action="store_true", help="time the staged (one call per stage) path instead of the fused one")
    ap.add_argument("--no-graph", action="store_true", help="fused path without CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (float32 / float64, under 64 MB in all; a "
                         "larger output as a fixed seeded sample of its rows, indices in DIR/<name>_rows.npy); N>1: DIR/rank<r>/")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    cfg = dict(CONFIGS[args.config])
    Z, H, W = (int(v) for v in args.shape.split(",")) if args.shape else cfg["shape"]
    if args.shape:
        cfg.pop("sides", None)
        cfg["name"] = "custom shape"
    if args.impl == "reference":
        run_reference(args, Z, H, W, cfg)
    else:
        run_ours(args, Z, H, W, cfg)


if __name__ == "__main__":
    main()
