#!/usr/bin/env python
"""The reference's strong-Dirichlet demo on the GPU (background-mesh mode):

    python demo/strong_dirichlet_flower.py [--n 200] [--degree 1] [--cell-type triangle|quadrilateral]

mirrors reference demo/strong-dirichlet/flower/main.py (`python main.py bg`) step by step -- background mesh of
[-4.5, 4.5]^2 (main.py:47-49), tags from the non-smooth detection level set (:52-64), phi-FEM forms with the
smooth level set (:85-131), solve (:138-157), u_h = phi_h w_h (:159-165) -- with the dolfinx / PETSc calls
replaced by phifem_b200 (INTEGRATION.md).  Prints the timings of each stage and a summary of the solution.
--cell-type quadrilateral runs the same steps on n^2 quadrilaterals of the same box (Q1 fields and level set; a Q2 trial
space is not implemented on quadrilaterals)."""
import argparse
import os
import sys
import time
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phifem_b200 import assemble, fem, solve, synthetic  # noqa: E402
from phifem.mesh_scripts import compute_tags_measures  # noqa: E402  (the reference's import line)


def main(n=200, degree=1, quiet=False, cell_type="triangle"):
    if cell_type not in ("triangle", "quadrilateral"):
        raise ValueError("cell_type must be 'triangle' or 'quadrilateral'")
    if cell_type == "quadrilateral" and degree != 1:
        raise ValueError("the strong-Dirichlet operator on quadrilaterals implements degree 1 (Q1) only")
    t = [time.perf_counter()]

    def lap(label):
        torch.cuda.synchronize()
        t.append(time.perf_counter())
        if not quiet:
            print("%-28s %8.2f ms" % (label, (t[-1] - t[-2]) * 1e3))

    make_mesh = synthetic.quadrilateral_mesh if cell_type == "quadrilateral" else synthetic.rectangle_mesh
    bg_mesh = make_mesh(n, lo=(-4.5, -4.5), hi=(4.5, 4.5))
    levelset_space = fem.functionspace(bg_mesh, ("Lagrange", 1))
    detection_levelset_h = fem.Function(levelset_space).interpolate(synthetic.flower_detection)
    lap("mesh + detection level set")
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        cells_tags, facets_tags, _, ds_bdy, _ = compute_tags_measures(bg_mesh, detection_levelset_h, 1,
                                                                      box_mode=True)
    ds = ds_bdy(100)
    lap("compute_tags_measures")
    primal_space = fem.functionspace(bg_mesh, ("Lagrange", degree))
    phi_space = fem.functionspace(bg_mesh, ("Lagrange", degree))
    phi_h = fem.Function(phi_space).interpolate(synthetic.flower_levelset)
    f_h = fem.Function(primal_space).interpolate(synthetic.flower_source)
    lap("interpolation (host)")
    plan = assemble.build_plan(bg_mesh, cells_tags, facets_tags, ds, V=primal_space, V_phi=phi_space)
    lap("symbolic phase")
    A, b = assemble.assemble_strong_dirichlet(plan, phi_h, f_h, stab_coef=1.0)
    lap("assembly (numeric)")
    w_h, info = solve.bicgstab(A, b, rtol=1e-10)
    if not info.converged:
        raise RuntimeError("the linear solve did not converge: %r" % info)
    lap("Jacobi-BiCGStab")
    phi_dev = torch.as_tensor(phi_h.x.array, device=w_h.device)
    u_h = w_h * phi_dev                      # main.py:165 (same space for w, phi and u here)
    if not quiet:
        print("cells %d (inside %d, cut %d), dofs %d, nnz %d" % (
            bg_mesh.num_cells, len(cells_tags.find(1)), len(cells_tags.find(2)), plan.n_rows, plan.nnz))
        print(info)
        print("u_h: min %.4e max %.4e" % (float(u_h.min()), float(u_h.max())))
    return u_h, info


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=200)
    ap.add_argument("--degree", type=int, default=1, choices=[1, 2])
    ap.add_argument("--cell-type", default="triangle", choices=["triangle", "quadrilateral"])
    a = ap.parse_args()
    if a.cell_type == "quadrilateral" and a.degree != 1:
        ap.error("--degree 2 is not implemented with --cell-type quadrilateral")
    main(a.n, a.degree, cell_type=a.cell_type)
