#!/usr/bin/env python3
"""Cost of splitting a mesh into its connected bodies on the device (engine.mesh_bodies, csrc/t3d_label.cu; DESIGN.md §4).

Meshes: the C1 phantom (512 x 1024^2 through pipeline.reconstruct_fused, one body), the C4-slab phantom (512 x 4096^2, one
body: the union-find's worst case is one root shared by every face) and the mesh of uniform noise (128 x 1024^2 at density
0.1, unsmoothed: many small bodies).  For each, with CUDA events over repeated calls after warm-up:
  * bodies: mesh_bodies on a mesh with nothing memoised (label + stats, with their host reads of B and of the largest term);
  * select: Bodies.select of the largest body (sizes from the host counts, no device read).
The device name and power limit are read in the same run.  Prints one JSON document and writes it to --out if given.

    python tools/bodies_bench.py --out profiles/r03_bodies_c1_c4slab_noise.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C1_phantom": ((512, 1024, 1024), "phantom"),
    "C4slab_phantom": ((512, 4096, 4096), "phantom"),
    "noise0.1_128x1024x1024": ((128, 1024, 1024), "noise"),
}


def power_limit():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                        str(__import__("torch").cuda.current_device())], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def timed(fn, reps, warmup):
    import torch
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def make_mesh(shape, kind):
    import numpy as np
    import torch
    from bench import PHYS, THRESHOLD, make_phantom_u8, side_counts
    from tomography_3d_reconstructor_b200 import engine, pipeline
    Z, H, W = shape
    dev = torch.device("cuda", torch.cuda.current_device())
    if kind == "phantom":
        u8 = make_phantom_u8(Z, H, W, 0, Z, dev)
        out = pipeline.reconstruct_fused(u8, THRESHOLD, side_counts(Z), PHYS["total_depth_mm"], PHYS["x_length_mm"],
                                         PHYS["y_length_mm"])
        mesh = out["mesh"]
    else:
        g = torch.Generator(device=dev)
        g.manual_seed(1234)
        u8 = (torch.rand((Z, H, W), device=dev, generator=g) < 0.1).to(torch.uint8)
        mesh = engine.extract_surface(engine.pack(u8, 1), np.full(Z, 6.0 / Z), PHYS["y_length_mm"] / H, PHYS["x_length_mm"] / W)
    mesh = engine.DeviceMesh(mesh.verts.contiguous(), mesh.faces.contiguous())
    del u8
    torch.cuda.empty_cache()
    return mesh


def run(name, reps, warmup):
    import numpy as np
    import torch
    from tomography_3d_reconstructor_b200 import engine
    shape, kind = WORKLOADS[name]
    mesh = make_mesh(shape, kind)

    def bodies():
        mesh._bodies = None
        return engine.mesh_bodies(mesh)

    t_bodies = timed(bodies, reps, warmup)
    b = bodies()
    fc = b.face_counts()
    keep = engine.component_keep(fc, 1, 1) - 1
    t_sel = timed(lambda: b.select(keep), reps, warmup)
    V, F = int(mesh.verts.shape[0]), int(mesh.faces.shape[0])
    res = {
        "workload": name, "shape": list(shape), "vertices": V, "faces": F, "bodies": b.n,
        "largest_body_faces": int(fc.max()) if len(fc) else 0, "bodies_ms": t_bodies, "select_ms": t_sel,
        "bodies_mfaces_per_s": F / t_bodies / 1e3, "reps": reps, "warmup": warmup,
    }
    del b, mesh
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--workloads", nargs="+", default=list(WORKLOADS), choices=list(WORKLOADS))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bodies_bench.py measures on a CUDA device; none is available")
    doc = {"device": torch.cuda.get_device_name(), "power_limit": power_limit(),
           "results": [run(w, args.reps, args.warmup) for w in args.workloads]}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
