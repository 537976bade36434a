#!/usr/bin/env python
"""Timing of the mixed-space operators beside the headline path (not the bench.py contract: one JSON line per operator).

    python tools/bench_operators.py [--ops neumann,neumann-quad,strong-quad,elasticity-2d,elasticity-3d] [--steps 10]
                                    [--warmup 3]

  neumann        BASELINE.json configs[1]: demo/neumann forms on a synthetic 4 M-cell triangle mesh (n = 1414), disc
  neumann-quad   the same forms on the demo's cell type: 2 M quadrilaterals on the same 2 M vertices (n = 1414), same
                 disc, Q2 level set (as the demo, levelset_degree = 2)
  strong-quad    demo/strong-dirichlet forms on the same 2 M quadrilaterals and disc: Q1 w, Q2 level set
  elasticity-2d  BASELINE.json configs[3] forms on 2 M triangles of the demo's box [-1.5, 1.5]^2 (n = 1000), unit disc
  elasticity-3d  BASELINE.json configs[3] as stated ("3D tetra mesh"): 384 000 Kuhn tetrahedra (n = 40), sphere

One step = cell tags + facet tags + zeroing + assembly (all kernels of the operator) on resident inputs, timed with CUDA
events on the launching stream; the symbolic phase (plan) is built once and timed separately.
"""
import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phifem_b200 import assemble, assemble_pk, elasticity, fem, mesh_scripts, synthetic  # noqa: E402
from phifem_b200.mesh import Measure, MeshTags  # noqa: E402


SYMMETRIC_BC = True   # --full-bc: the pass over the whole matrix instead of the list-driven one (phifem_apply_dirichlet_symmetric)


def _tags(mesh, phi):
    # quadrilaterals: the tag kernels gather the level set through a dofmap, which only the full space carries
    V = fem.functionspace(mesh, 1) if mesh.cell_type == "quadrilateral" else fem.functionspace_p1_device(mesh)
    dls = mesh_scripts._DeviceLevelset(mesh, fem.Function(V, phi), 1)
    ws = mesh_scripts.TagWorkspace(mesh)
    mesh_scripts.classify(mesh, dls, ws=ws)
    tdim = mesh.topology.dim
    ctags, ftags = MeshTags(mesh, tdim, ws.cell_tags), MeshTags(mesh, tdim - 1, ws.facet_tags)
    ctags.tags8, ftags.tags8 = ws.cell_tags8, ws.facet_tags8
    e100 = mesh_scripts._integration_entities_dev(mesh, ws.cell_tags8, ws.facet_tags8, 4, (1, 2))
    e101 = mesh_scripts._integration_entities_dev(mesh, ws.cell_tags8, ws.facet_tags8, 3, (2, 3))
    return dls, ws, ctags, ftags, Measure("ds", mesh, subdomain_data=[(100, e100), (101, e101)])


def _time(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    ms = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(steps))
    return ev[0].elapsed_time(ev[-1]) / steps, ms[0]


def run(op, steps, warmup):
    dev = torch.device("cuda", 0)
    t0 = time.perf_counter()
    if op in ("neumann", "neumann-quad", "strong-quad"):
        n = 1414
        mesh = (synthetic.rectangle_mesh if op == "neumann" else synthetic.quadrilateral_mesh)(n, device=dev)
        phi = synthetic.sphere_levelset(mesh.x, center=(0.0031, 0.0027), radius=0.6)
    elif op == "elasticity-2d":
        n = 1000
        mesh = synthetic.rectangle_mesh(n, lo=(-1.5, -1.5), hi=(1.5, 1.5), device=dev)
        phi = 1.0 - ((mesh.x[:, 0] - 0.0031) ** 2 + (mesh.x[:, 1] - 0.0027) ** 2)
    else:
        n = 40
        mesh = synthetic.box_mesh(n, device=dev)
        phi = synthetic.sphere_levelset(mesh.x)
    mesh.c2f
    if mesh.cell_type != "quadrilateral":
        mesh.detj_bounds()
    dls, ws, ctags, ftags, ds = _tags(mesh, phi)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    g = torch.Generator(device="cpu").manual_seed(1234)
    if op in ("neumann", "neumann-quad"):
        V_phi = fem.functionspace(mesh, 2) if op == "neumann-quad" else None
        plan = assemble.build_plan_neumann(mesh, ctags, ftags, ds(100), V_phi=V_phi)
        phi_a = phi if V_phi is None else synthetic.sphere_levelset(V_phi.dof_coordinates_dev(),
                                                                    center=(0.0031, 0.0027), radius=0.6)
        f = (2 * torch.rand(mesh.num_vertices, generator=g, dtype=torch.float64) - 1).to(dev)
        un = (2 * torch.rand(mesh.num_vertices, generator=g, dtype=torch.float64) - 1).to(dev)
        data, b = plan.new_outputs()
        asm = lambda: assemble_pk.assemble_neumann_into(plan, phi_a, f, un, 1.0, 1.0, data, b)   # noqa: E731
    elif op == "strong-quad":
        V_phi = fem.functionspace(mesh, 2)
        plan = assemble.build_plan(mesh, ctags, ftags, ds(100), V_phi=V_phi)
        phi_a = synthetic.sphere_levelset(V_phi.dof_coordinates_dev(), center=(0.0031, 0.0027), radius=0.6)
        f = (2 * torch.rand(mesh.num_vertices, generator=g, dtype=torch.float64) - 1).to(dev)
        data, b = plan.new_outputs()
        asm = lambda: assemble_pk.assemble_pk_into(plan, phi_a, f, 1.0, data, b)   # noqa: E731
    else:
        plan = elasticity.build_plan_interface_elasticity(mesh, ctags, ftags, ds)
        f = (2 * torch.rand(mesh.num_vertices, mesh.gdim, generator=g, dtype=torch.float64) - 1).to(dev)
        mat = elasticity.Material()
        bv = plan.boundary_vertices()
        marker = torch.zeros(plan.n_rows, dtype=torch.int8, device=dev)
        values = torch.zeros(plan.n_rows, dtype=torch.float64, device=dev)
        bc_dofs = plan.dofs("u_in", bv).reshape(-1)
        marker[bc_dofs] = 1
        bc_list = bc_dofs.to(torch.int32).contiguous() if SYMMETRIC_BC else None
        data, b = plan.new_outputs()
        asm = lambda: elasticity.assemble_interface_elasticity_into(plan, phi, f, mat, 1.0, 1.0, data, b,   # noqa: E731
                                                                   marker, values, bc_list)
    torch.cuda.synchronize()
    t2 = time.perf_counter()

    def tags_step():
        mesh_scripts.classify_cells(mesh, dls, ws)
        mesh_scripts.classify_facets(mesh, dls, ws)

    def step():
        tags_step()
        asm()

    ms, ms_min = _time(step, steps, warmup)
    ms_tags, _ = _time(tags_step, steps, warmup)
    ms_asm, _ = _time(asm, steps, warmup)
    c8 = ws.cell_tags8
    line = {"operator": op, "metric": "phi-FEM cells assembled/s (tags+CSR)", "value": mesh.num_cells / (ms * 1e-3),
            "unit": "cells/s", "ms_per_step": ms, "ms_min": ms_min, "ms_tags": ms_tags, "ms_assembly": ms_asm,
            "steps": steps, "warmup": warmup, "dtype": "f64", "data": "synthetic",
            "config": {"n": n, "cells": mesh.num_cells, "vertices": mesh.num_vertices,
                       "interior": int((c8 == 1).sum()), "cut": int((c8 == 2).sum()), "exterior": int((c8 == 3).sum()),
                       "rows": plan.n_rows, "nnz": plan.nnz},
            "csr_write_gbs": 8.0 * plan.nnz / (ms_asm * 1e-3) / 1e9,
            "dirichlet_pass": ("list" if SYMMETRIC_BC else "full") if op.startswith("elasticity") else None,
            "topology_s": t1 - t0, "symbolic_s": t2 - t1}
    print(json.dumps(line), flush=True)
    return line


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ops", default="neumann,elasticity-2d,elasticity-3d")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--full-bc", action="store_true")
    a = ap.parse_args()
    SYMMETRIC_BC = not a.full_bc
    for name in a.ops.split(","):
        run(name, a.steps, a.warmup)
        torch.cuda.empty_cache()
