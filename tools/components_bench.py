#!/usr/bin/env python3
"""Cost of device connected-component labelling (engine.label_components, csrc/t3d_label.cu; DESIGN.md §4).

Workloads: the C1 ellipsoid phantom (512 x 1024^2, one run per row), C1 uniform noise at density 0.3 with 6- and with
26-connectivity (runs everywhere; near the 6-connected percolation threshold, one giant component at 26), and the C4-slab
phantom (512 x 4096^2).  For each it times, with CUDA events over repeated calls after warm-up:
  * label: count + label + stats, i.e. label_components on a fresh volume (two host reads of R and K inside);
  * volumes: Components.volumes_mm3; expand: the int32 label volume; select: the grid of the largest component.
The device name and power limit are read in the same run.  Prints one JSON document and writes it to --out if given.

    python tools/components_bench.py --out profiles/r03_components_c1_c4slab.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "C1_phantom_6": ((512, 1024, 1024), "phantom", 6),
    "C1_noise0.3_6": ((512, 1024, 1024), "noise", 6),
    "C1_noise0.3_26": ((512, 1024, 1024), "noise", 26),
    "C4slab_phantom_6": ((512, 4096, 4096), "phantom", 6),
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


def make_volume(shape, kind):
    import torch
    from bench import THRESHOLD, make_phantom_u8
    from tomography_3d_reconstructor_b200 import engine
    Z, H, W = shape
    dev = torch.device("cuda", torch.cuda.current_device())
    if kind == "phantom":
        u8 = make_phantom_u8(Z, H, W, 0, Z, dev)
        dv = engine.pack(u8, THRESHOLD)
    else:
        g = torch.Generator(device=dev)
        g.manual_seed(1234)
        u8 = (torch.rand((Z, H, W), device=dev, generator=g) < 0.3).to(torch.uint8)
        dv = engine.pack(u8, 1)
    del u8
    torch.cuda.empty_cache()
    return dv


def run(name, reps, warmup):
    import numpy as np
    import torch
    from tomography_3d_reconstructor_b200 import engine
    shape, kind, conn = WORKLOADS[name]
    dv = make_volume(shape, kind)
    Z, H, W = shape

    def label():
        dv.memo.clear()
        return engine.label_components(dv, conn)

    t_label = timed(label, reps, warmup)
    comps = label()
    depths = np.full(Z, 6.0 / Z)
    t_vol = timed(lambda: comps.volumes_mm3(0.14, 0.093, depths), reps, warmup)
    counts = comps.counts()
    keep = engine.component_keep(counts, 1, 1)
    t_sel = timed(lambda: comps.select(keep), reps, warmup)
    t_exp = timed(comps.labels, reps, warmup)
    vox = Z * H * W
    res = {
        "workload": name, "shape": list(shape), "connectivity": conn, "voxels": vox, "set_voxels": int(counts.sum()),
        "runs": comps.n_runs, "components": comps.n, "largest_component": int(counts.max()) if len(counts) else 0,
        "label_ms": t_label, "volumes_ms": t_vol, "expand_ms": t_exp, "select_ms": t_sel,
        "label_gvoxel_per_s": vox / t_label / 1e6, "label_mruns_per_s": comps.n_runs / t_label / 1e3,
        "expand_write_gb_per_s": 4 * vox / t_exp / 1e6, "select_gvoxel_per_s": vox / t_sel / 1e6,
        "reps": reps, "warmup": warmup,
    }
    del comps, dv
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
        raise SystemExit("components_bench.py measures on a CUDA device; none is available")
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
