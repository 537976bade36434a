#!/usr/bin/env python
"""Build time of the interface-elasticity symbolic phase: the torch `ElasticityPlan` against the device builder behind
the C ABI (`phifem_elasticity_pattern_create`, through `symbolic.DeviceElasticityPattern`), at pattern sizes near the
int32 limit of the blocked CSR.

    python tools/time_symbolic_elasticity.py [--reps 3] [--out FILE.jsonl]

Problems (P1 level set, P1 detection, box mode):
  - tri:  rectangle_mesh(1000), bench's disc DISC_CENTER / DISC_RADIUS (about 1.0 M vertices, 1.4e9 blocked entries);
  - quad: quadrilateral_mesh(800), the same disc;
  - tet:  box_mesh(48), bench's sphere (about 1.3e9 blocked entries).
Both builders get the same resident inputs (tags, ds(100) / ds(101) entities); each call is timed with a host clock up
to a device synchronisation.  After one warm-up call of each, the two alternate `--reps` times; the best is reported.
A last native call runs under torch.profiler, apart from the timed ones, for the time of the blocked-CSR expansion
kernel (k_expand_blocks): its bytes written (4 per blocked entry) over that time, against the 7.7 TB/s of the data
sheet.  Every line records the card's name and power limit, and whether the two builders' arrays are equal.
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
from phifem_b200 import assemble, elasticity, fem, mesh_scripts, symbolic, synthetic  # noqa: E402

NAMES = ("vptr", "indptr", "indices", "cut_cells", "facets_in", "facets_out", "entities_in", "entities_out",
         "pos_cells", "pos_facets_in", "pos_facets_out", "pos_entities_in", "pos_entities_out")
PEAK_BYTES_PER_S = 7.7e12
SIZES = {"tri": 1000, "quad": 800, "tet": 48}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, check=True)
        name, power = [s.strip() for s in q.stdout.strip().split(",")]
    except (OSError, subprocess.CalledProcessError, ValueError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def problem(name):
    n = SIZES[name]
    if name == "tet":
        mesh, ls_kw = synthetic.box_mesh(n, device="cuda"), {}
    else:
        make = synthetic.rectangle_mesh if name == "tri" else synthetic.quadrilateral_mesh
        mesh, ls_kw = make(n, device="cuda"), dict(center=bench.DISC_CENTER, radius=bench.DISC_RADIUS)
    V1 = fem.functionspace(mesh, 1)
    det = fem.Function(V1, synthetic.sphere_levelset(mesh.x, **ls_kw))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        ctags, ftags, _, d_bdry, _ = mesh_scripts.compute_tags_measures(mesh, det, 1, box_mode=True)
    c8, f8, e_in = assemble._plan_inputs(mesh, ctags, ftags, d_bdry(100))
    _, _, e_out = assemble._plan_inputs(mesh, ctags, ftags, d_bdry(101))
    V1.dofmap_dev
    mesh.f2c
    if mesh.cell_type != "quadrilateral":
        mesh.boundary_records()                             # per-mesh records outside the timing
    return n, mesh, V1, ctags, ftags, (e_in, e_out), c8, f8


def timed(fn):
    torch.cuda.synchronize()
    t = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, (time.perf_counter() - t) * 1e3


def expansion_kernel_ms(native):
    """Device time of k_expand_blocks in one native call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pat = native()
        torch.cuda.synchronize()
    del pat
    us = [e.device_time_total for e in prof.events() if "k_expand_blocks" in e.name]
    return sum(us) / 1e3 if us else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--problems", default="tri,quad,tet")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu, power = card()
    lines = []
    for name in args.problems.split(","):
        n, mesh, V1, ctags, ftags, ents, c8, f8 = problem(name)
        torch_plan = lambda: elasticity.ElasticityPlan(mesh, c8, f8, ents[0], ents[1], V1)  # noqa: E731
        native = lambda: symbolic.DeviceElasticityPattern(mesh, ctags, ftags, ents)      # noqa: E731
        ref, _ = timed(torch_plan)                                                       # warm-up, reference arrays
        pat, _ = timed(native)                                                           # warm-up
        equal = pat.nnz == ref.nnz and all(torch.equal(getattr(pat, k), getattr(ref, k)) for k in NAMES)
        rec = {"problem": name, "n": n, "cell_type": mesh.cell_type, "vertices": mesh.num_vertices,
               "cells": mesh.num_cells, "nb": ref.nb, "n_rows": ref.n_rows, "vertex_pairs": int(ref.vptr[-1]),
               "nnz": ref.nnz, "n_cut": int(ref.cut_cells.numel()), "n_facets_in": int(ref.facets_in.numel()),
               "n_facets_out": int(ref.facets_out.numel()), "n_entities_in": int(ref.entities_in.shape[0]),
               "n_entities_out": int(ref.entities_out.shape[0]), "arrays_equal": bool(equal)}
        del pat, ref
        torch.cuda.empty_cache()
        ms = {"torch": [], "native": []}
        for _ in range(args.reps):
            for kind, fn in (("torch", torch_plan), ("native", native)):
                out, t = timed(fn)
                ms[kind].append(t)
                del out
                torch.cuda.empty_cache()
        kms = expansion_kernel_ms(native)
        written = 4 * rec["nnz"]
        rec.update({"torch_ms": min(ms["torch"]), "native_ms": min(ms["native"]), "torch_ms_all": ms["torch"],
                    "native_ms_all": ms["native"], "expansion_kernel_ms": kms, "expansion_bytes_written": written,
                    "expansion_tb_per_s": written / kms / 1e9 if kms else None,
                    "expansion_share_of_7_7_tb_per_s": written / kms / 1e-3 / PEAK_BYTES_PER_S if kms else None,
                    "gpu": gpu, "power_limit": power})
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        del mesh, V1, ctags, ftags, ents, c8, f8
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
