#!/usr/bin/env python
"""Device-resident classification of hexahedral meshes beside tetrahedral meshes on the same vertices.

    python tools/bench_hex_tags.py [--n 100,200] [--steps 20] [--warmup 3] [--out FILE.jsonl]

For every n: `synthetic.hexahedron_mesh(n)` (n^3 cells) and `synthetic.box_mesh(n)` (6 n^3 Kuhn tetrahedra) share
their (n + 1)^3 vertices and the sphere level set of bench.py (Q1 / P1 vertex values, detection degree 1).  One step =
cell tags + facet tags (`mesh_scripts.classify`, no host synchronisation) on resident inputs, timed with CUDA events;
the two meshes alternate, `--reps` rounds each.  The tetrahedra take the P1 fast path, the hexahedra the generic
table-driven kernels (csrc/tags.cu).  Prints one JSON line per (n, cell type), with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phifem_b200 import fem, mesh_scripts, synthetic  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, check=True)
        name, power = [s.strip() for s in q.stdout.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def setup(mesh):
    phi = synthetic.sphere_levelset(mesh.x)
    V = fem.functionspace_p1_device(mesh) if mesh.cell_type == "tetrahedron" else fem.functionspace(mesh, 1)
    dls = mesh_scripts._DeviceLevelset(mesh, fem.Function(V, phi), 1)
    ws = mesh_scripts.TagWorkspace(mesh)
    return dls, ws


def time_steps(mesh, dls, ws, steps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        mesh_scripts.classify(mesh, dls, ws=ws)
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="100,200")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, power = card()
    lines = []
    for n in (int(s) for s in args.n.split(",")):
        meshes = {"hexahedron": synthetic.hexahedron_mesh(n), "tetrahedron": synthetic.box_mesh(n)}
        state = {}
        for ct, mesh in meshes.items():
            mesh.f2c, mesh.boundary_facets, mesh.detj_bounds()   # topology and per-mesh records outside the timing
            state[ct] = setup(mesh)
            time_steps(mesh, *state[ct], args.warmup)
        ms = {ct: [] for ct in meshes}
        for _ in range(args.reps):
            for ct, mesh in meshes.items():
                ms[ct].append(time_steps(mesh, *state[ct], args.steps))
        for ct, mesh in meshes.items():
            ws = state[ct][1]
            tags = torch.bincount(ws.cell_tags8.long(), minlength=4).cpu().tolist()
            rec = {"n": n, "cell_type": ct, "cells": mesh.num_cells, "facets": mesh.num_facets,
                   "vertices": mesh.num_vertices, "cell_tag_counts": tags[1:4], "ms_per_classify": min(ms[ct]),
                   "ms_all_reps": ms[ct], "steps": args.steps, "gpu": name, "power_limit": power}
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
        del meshes, state
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
