#!/usr/bin/env python
"""Build time of the quadrature-kernel symbolic phase: the torch `PkAssemblyPlan` against the device builder behind the
C ABI (`phifem_pk_pattern_create`, through `symbolic.DevicePkPattern`), on the problems of bench.py.

    python tools/time_symbolic_pk.py [--reps 3] [--out FILE.jsonl]

Problems (bench.py's sizes, level sets and tags; P1 detection):
  - 2d-p2: rectangle_mesh(CONFIGS["2d-p2"] n), disc DISC_CENTER / DISC_RADIUS, strong Dirichlet, P2 / P2;
  - 3d-p2: box_mesh(CONFIGS["3d-p2"] n), bench's sphere, strong Dirichlet, P2 / P2;
  - 2d-p1-weak: rectangle_mesh(CONFIGS["2d-p1"] n), the disc, the weak-Dirichlet operator, P1 / P1.
Both builders get the same resident inputs (tags, ds(100) entities, the plan's pattern dofmap); each call is timed with
a host clock up to a device synchronisation.  After one warm-up call of each, the two alternate `--reps` times; the
best is reported.  Every line records the card's name and power limit, and whether the two builders' arrays are equal.
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from phifem_b200 import assemble, fem, mesh_scripts, symbolic, synthetic  # noqa: E402
from phifem_b200.assemble_pk import PkAssemblyPlan  # noqa: E402

NAMES = ("indptr", "indices", "active", "cut_positions", "ghost", "entities", "slots_cells", "slots_ghost",
         "slots_boundary")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, check=True)
        name, power = [s.strip() for s in q.stdout.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def problem(name):
    if name == "3d-p2":
        n = bench.CONFIGS["3d-p2"][0]
        mesh, ls_kw, form, degree = synthetic.box_mesh(n, device="cuda"), {}, "strong", 2
    else:
        config = "2d-p2" if name == "2d-p2" else "2d-p1"
        n = bench.CONFIGS[config][0]
        mesh = synthetic.rectangle_mesh(n, device="cuda")
        ls_kw = dict(center=bench.DISC_CENTER, radius=bench.DISC_RADIUS)
        form, degree = ("strong", 2) if name == "2d-p2" else ("weak", 1)
    det = fem.Function(fem.functionspace(mesh, 1), synthetic.sphere_levelset(mesh.x, **ls_kw))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, ds, _ = mesh_scripts.compute_tags_measures(mesh, det, 1, box_mode=True)
    V = fem.functionspace(mesh, degree)
    V.dofmap_dev
    c8, f8, ents = assemble._plan_inputs(mesh, ctags, ftags, ds(100))
    mesh.f2c, mesh.boundary_records()                       # per-mesh records outside the timing
    return n, mesh, V, ctags, ftags, ds(100), c8, f8, ents, form


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--problems", default="2d-p2,3d-p2,2d-p1-weak")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu, power = card()
    lines = []
    for name in args.problems.split(","):
        n, mesh, V, ctags, ftags, ds100, c8, f8, ents, form = problem(name)
        torch_plan = lambda: PkAssemblyPlan(mesh, c8, f8, ents, V, V, form=form)  # noqa: E731
        ref, _ = timed(torch_plan)                                               # warm-up, and the reference arrays
        native = lambda: symbolic.DevicePkPattern(mesh, ctags, ftags, ds100, ref.pattern_dofmap, ref.n_rows)  # noqa
        pat, _ = timed(native)                                                   # warm-up
        equal = pat.nnz == ref.nnz and all(torch.equal(getattr(pat, k), getattr(ref, k)) for k in NAMES)
        rec = {"problem": name, "n": n, "cells": mesh.num_cells, "form": form, "degree": V.degree,
               "pattern_dofs_per_cell": int(ref.pattern_dofmap.shape[1]), "n_rows": ref.n_rows, "nnz": ref.nnz,
               "n_active": int(ref.active.numel()), "n_ghost": int(ref.ghost.numel()),
               "n_entities": int(ref.entities.shape[0]), "arrays_equal": bool(equal)}
        del pat
        ms = {"torch": [], "native": []}
        for _ in range(args.reps):
            for kind, fn in (("torch", torch_plan), ("native", native)):
                out, t = timed(fn)
                ms[kind].append(t)
                del out
        rec.update({"torch_ms": min(ms["torch"]), "native_ms": min(ms["native"]), "torch_ms_all": ms["torch"],
                    "native_ms_all": ms["native"], "gpu": gpu, "power_limit": power})
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        del ref, mesh, V, ctags, ftags, ds100, c8, f8, ents
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
