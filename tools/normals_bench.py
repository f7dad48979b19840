#!/usr/bin/env python3
"""Cost of the field-gradient vertex normals in the fused step (DESIGN.md §4).

For each config (C1 = 512 x 1024^2, the C4 slab = 512 x 4096^2; ellipsoid phantom as in bench.py) it times, in one run:
  * the captured step of reconstruct_fused with normals off and on, alternating blocks of graph replays (CUDA events);
  * t3d_reconstruct_normals alone (tie pass + normals kernel), CUDA events around repeated launches on the step's state.
The device name and power limit are read in the same run.  Prints one JSON document and writes it to --out if given.

    python tools/normals_bench.py --configs C1 C4 --out profiles/r03_normals_c1_c4slab.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = {"C1": (512, 1024, 1024), "C4": (512, 4096, 4096)}


def power_limit():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                                        str(__import__("torch").cuda.current_device())], text=True).strip()
    except (OSError, subprocess.CalledProcessError):
        return "unknown"


def time_replays(plan, n):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        plan.graph.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def run_config(name, rounds, per_block, launches):
    import numpy as np
    import torch
    from bench import PHYS, THRESHOLD, make_phantom_u8, side_counts
    from tomography_3d_reconstructor_b200 import engine, pipeline
    Z, H, W = SHAPES[name]
    masks = make_phantom_u8(Z, H, W, 0, Z, torch.device("cuda", torch.cuda.current_device()))
    sides = side_counts(Z)
    phys = (PHYS["total_depth_mm"], PHYS["x_length_mm"], PHYS["y_length_mm"])
    plans = {}
    for normals in (False, True):
        for _ in range(3):                     # staged first call, capture, one replay
            out = pipeline.reconstruct_fused(masks, THRESHOLD, sides, *phys, normals=normals)
        key = pipeline.plan_key(masks, THRESHOLD, sides, *phys, normals=normals)
        plans[normals] = pipeline._plans[key]
        assert plans[normals].graph is not None, "the fused plan did not run"
    n_verts = int(out["mesh"].verts.shape[0])
    nrm = out["normals"]
    unit_err = float((torch.linalg.vector_norm(nrm.double(), dim=1) - 1).abs().max())
    step = {False: [], True: []}
    for _ in range(rounds):
        for normals in (False, True):
            step[normals].append(time_replays(plans[normals], per_block))
    # the post-step alone, on the state the last replay of the normals plan left behind
    p = plans[True]
    L = engine._L()
    time_replays(p, 1)

    def enqueue_normals():
        engine.check(L.t3d_reconstruct_normals(
            Z, H, W, p.n_stages, p.erode_mask, 1 if p.add_padding else 0, engine._W3_C, engine._p(p.adj_d), p.n_cum,
            float(p.mm_y), float(p.mm_x), *p.caps, engine._p(p.res), engine._p(p.ws), engine._p(p.normals), engine._stream()),
            "t3d_reconstruct_normals")

    enqueue_normals()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        enqueue_normals()
    b.record()
    b.synchronize()
    alone_ms = a.elapsed_time(b) / launches
    med = {k: float(np.median(v)) for k, v in step.items()}
    res = {
        "config": name, "shape": [Z, H, W], "vertices": n_verts, "normal_unit_error_max": unit_err,
        "step_ms_normals_off_median": med[False], "step_ms_normals_on_median": med[True],
        "step_ms_normals_off_blocks": step[False], "step_ms_normals_on_blocks": step[True],
        "normals_delta_ms": med[True] - med[False],
        "normals_entry_ms": alone_ms, "normals_entry_ns_per_vertex": 1e6 * alone_ms / max(n_verts, 1),
        "replays_per_block": per_block, "blocks": rounds, "entry_launches": launches,
    }
    pipeline._plans.clear()
    pipeline._hints.clear()
    del masks, plans, p, out, nrm
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--configs", nargs="+", default=["C1", "C4"], choices=sorted(SHAPES))
    ap.add_argument("--rounds", type=int, default=6, help="alternating blocks per mode")
    ap.add_argument("--replays", type=int, default=10, help="graph replays per block (>= 20 per mode in all)")
    ap.add_argument("--launches", type=int, default=50, help="launches of t3d_reconstruct_normals timed together")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("normals_bench.py measures on a CUDA device; none is available")
    doc = {"device": torch.cuda.get_device_name(), "power_limit": power_limit(),
           "results": [run_config(c, args.rounds, args.replays, args.launches) for c in args.configs]}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
