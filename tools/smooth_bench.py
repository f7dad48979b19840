#!/usr/bin/env python3
"""Cost of smoothing a mesh on the device (engine.vertex_neighbors / engine.smooth_mesh, csrc/t3d_smooth.cu; DESIGN.md §4).

Meshes: as tools/bodies_bench.py, the C1 phantom (512 x 1024^2 through pipeline.reconstruct_fused), the C4-slab phantom
(512 x 4096^2) and the mesh of uniform noise (128 x 1024^2 at density 0.1, unsmoothed: the most ambiguous cubes and the
longest rows).  For each, with CUDA events over repeated calls after warm-up:
  * adjacency: vertex_neighbors on a mesh with nothing memoised (count, the host read of N, emit);
  * taubin_1: smooth_mesh with one iteration (adjacency memoised; one launch, float32 in and out);
  * taubin_10: smooth_mesh at trimesh's defaults (10 iterations, lamb = nu = 0.5);
  * per_iteration: (taubin_10 - taubin_1) / 9, one float64 -> float64 step;
  * bytes per iteration: offsets, neighbour ids, one read and one write of the positions (float64), the least a step moves;
    the neighbour gathers (degree x 24 B per vertex) come from L2 and are counted apart.
The device name and power limit are read in the same run.  Prints one JSON document and writes it to --out if given.

    python tools/smooth_bench.py --out profiles/r03_smooth_c1_c4slab_noise.json
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bodies_bench import WORKLOADS, make_mesh, power_limit, timed  # noqa: E402  same meshes, clock and card query


def run(name, reps, warmup):
    import torch
    from tomography_3d_reconstructor_b200 import engine
    shape, kind = WORKLOADS[name]
    mesh = make_mesh(shape, kind)

    def adjacency():
        mesh._adjacency = None
        return engine.vertex_neighbors(mesh)

    t_adj = timed(adjacency, reps, warmup)
    off, nb = adjacency()
    t1 = timed(lambda: engine.smooth_mesh(mesh, 1), reps, warmup)
    t10 = timed(lambda: engine.smooth_mesh(mesh), reps, warmup)
    V, F, N = int(mesh.verts.shape[0]), int(mesh.faces.shape[0]), int(nb.shape[0])
    per_it = (t10 - t1) / 9
    step_bytes = 8 * (V + 1) + 4 * N + 2 * 24 * V
    res = {
        "workload": name, "shape": list(shape), "vertices": V, "faces": F, "neighbours": N,
        "max_degree": int((off[1:] - off[:-1]).max()) if V else 0,
        "adjacency_ms": t_adj, "taubin_1_ms": t1, "taubin_10_ms": t10, "per_iteration_ms": per_it,
        "step_bytes": step_bytes, "step_gbytes_per_s": step_bytes / per_it / 1e6, "gather_bytes": 24 * N,
        "reps": reps, "warmup": warmup,
    }
    del off, nb, mesh
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
        raise SystemExit("smooth_bench.py measures on a CUDA device; none is available")
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
