#!/usr/bin/env python
"""Benchmark of the phi-FEM hot path: cut-cell tags + CSR assembly, cells/s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--n 204] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the synthetic 3D P1 configuration of BASELINE.json
(config E, SURVEY.md section 8d): classify all cells and facets of a 6 n^3 Kuhn-tetrahedra unit cube
against a sphere level set, then assemble the strong-Dirichlet phi-FEM operator and load vector into
CSR (pattern / slot maps are the precomputed symbolic phase, timed separately as `symbolic_ms`).
Prints ONE JSON line (rank 0).  `value` times the device-resident pass with CUDA events; `e2e` times
the public API with pinned host buffers for the level set, the source term and all results.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "phi-FEM cells assembled/s (tags+CSR)"
UNIT = "cells/s"
# 2D configurations (BASELINE.json configs[1..2], SURVEY.md 8d): disc in [-1, 1]^2, offsets keep |phi_v| >> ulp
DISC_CENTER = (3.141592653589793 / 1000.0, 2.718281828459045 / 1000.0)
DISC_RADIUS = 0.6
CONFIGS = {   # name -> (default n, description)
    "3d-p1": (204, "synthetic 3D P1 phi-FEM Poisson (BASELINE.json configs[4]): %d Kuhn tetrahedra per GPU "
                   "(n=%d), sphere level set"),
    "2d-p1": (1414, "synthetic 2D P1 phi-FEM Poisson (BASELINE.json configs[1] scale, 4 M triangles): %d "
                    "triangles (n=%d), disc level set"),
    "2d-p2": (2828, "synthetic 2D P2 phi-FEM Poisson (BASELINE.json configs[2], 16 M triangles): %d triangles "
                    "(n=%d), disc level set, P2 trial/test space and P2 level set, P1 detection"),
    "3d-p2": (64, "synthetic 3D P2 phi-FEM Poisson: %d Kuhn tetrahedra (n=%d), sphere level set, P2 trial/test "
                  "space and P2 level set, P1 detection"),
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {}
        for key in dir(nv):
            if key.startswith("nvmlClocksEventReason") or key.startswith("nvmlClocksThrottleReason"):
                val = getattr(nv, key)
                if isinstance(val, int) and val and "All" not in key and "None" not in key:
                    names.setdefault(val, key.replace("nvmlClocksEventReason", "")
                                     .replace("nvmlClocksThrottleReason", ""))
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if bits & bit and name not in ("GpuIdle", "ApplicationsClocksSetting"):
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def algorithmic_bytes(counts, tag_bytes=1):
    """SURVEY.md section 8(d): compulsory traffic, each input read once / each output written once.  tag_bytes: width of
    the tag arrays the kernels WRITE (1: the int8 arrays of the product path; 4: SURVEY's yardstick, the int32 arrays of
    the reference's MeshTags, which the product widens on demand and never writes in the timed region)."""
    nc, nv, nf, gdim, nvpc = counts["Nc"], counts["Nv"], counts["Nf"], counts["gdim"], counts["nvpc"]
    na, nva, ng, nnz = counts["Na"], counts["Nv_active"], counts["Ng"], counts["nnz"]
    nd, nrow = counts.get("nd", nvpc), counts.get("Nrow", nv)
    ndof_a = counts.get("Ndof_active", nva)          # active dofs of the trial/test space (= of phi and f)
    b_tags_cells = 4 * nvpc * nc + 8 * nv + tag_bytes * nc
    b_tags_facets = 4 * nvpc * nc + tag_bytes * nf    # c2f (== f2c in size) + facet tags out
    geo = 4 * nvpc * na if nd != nvpc else 0          # P2: cell -> vertex for the geometry besides the dofmap
    b_asm = (4 * nd * na + geo + 8 * gdim * nva + 8 * ndof_a + 8 * ndof_a + tag_bytes * na + 8 * ng + 12 * nnz
             + 4 * (nrow + 1) + 8 * nrow)
    # the numeric cell kernel alone: no column indices / indptr (they belong to the symbolic phase)
    b_cells_kernel = 4 * nd * na + geo + 8 * gdim * nva + 16 * ndof_a + tag_bytes * na + 8 * nnz + 8 * ndof_a
    return {"tags_cells": b_tags_cells, "tags_facets": b_tags_facets, "assembly": b_asm,
            "cells_kernel": b_cells_kernel, "total": b_tags_cells + b_tags_facets + b_asm}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (cpu_baseline of our line, and --impl reference)
# ------------------------------------------------------------------------------------------------
class CpuWorkload:
    """Tags + CSR assembly on host arrays with the C/OpenMP oracle port (oracle/csrc/phifem_oracle.c).  The symbolic
    phase (topology, pattern, slot maps) is SETUP, excluded from the timing like `symbolic_ms` of the GPU arm; it comes
    either from torch ops on CPU tensors (`from_size`: no GPU needed, small n) or from the arrays an already-built
    device plan holds (`from_device`: config E itself, n = 204)."""

    def __init__(self, x, cells, c2f, f2c, phi, f, plan_arrays, nnz, label):
        from oracle import native as ON
        self.ON = ON
        self.x, self.cells, self.c2f, self.f2c, self.phi, self.f = x, cells, c2f, f2c, phi, f
        self.plan, self.nnz, self.num_cells, self.label = plan_arrays, nnz, len(cells), label

    @classmethod
    def from_size(cls, n):
        import torch
        from oracle import native as ON
        from oracle import tags as OT
        from phifem_b200 import assemble, synthetic
        from phifem_b200.mesh import MeshTags
        mesh = synthetic.box_mesh(n, device="cpu")
        x = mesh.x.numpy()
        cells = np.ascontiguousarray(mesh.cells.numpy())
        c2f, f2c = np.ascontiguousarray(mesh.c2f.numpy()), np.ascontiguousarray(mesh.f2c.numpy())
        phi = synthetic.sphere_levelset(mesh.x).numpy()
        f = synthetic.ball_source(mesh.x).numpy()
        ct = ON.tag_cells_p1(x, cells, phi)
        ft = ON.tag_facets_p1(x, cells, c2f, f2c, phi, ct)
        ents = OT.integration_entities(c2f, f2c, (ct == 1) | (ct == 2), ft == 4)
        plan = assemble.build_plan(mesh, MeshTags(mesh, 3, torch.from_numpy(ct)),
                                   MeshTags(mesh, 2, torch.from_numpy(ft)), ents, method="atomic")
        arrays = {k: np.ascontiguousarray(getattr(plan, k).numpy())
                  for k in ("active", "slots_cells", "entities", "slots_boundary", "ghost", "slots_ghost")}
        return cls(x, cells, c2f, f2c, phi, f, arrays, plan.nnz, "n=%d Kuhn unit cube" % n)

    @classmethod
    def from_device(cls, mesh, phi, f, plan, n):
        arrays = {k: np.ascontiguousarray(getattr(plan, k).cpu().numpy())
                  for k in ("active", "slots_cells", "entities", "slots_boundary", "ghost", "slots_ghost")}
        host = lambda t: np.ascontiguousarray(t.cpu().numpy())     # noqa: E731
        return cls(host(mesh.x), host(mesh.cells), host(mesh.c2f), host(mesh.f2c), host(phi), host(f), arrays,
                   plan.nnz, "n=%d Kuhn unit cube" % n)

    def step(self):
        ON, p = self.ON, self.plan
        ct = ON.tag_cells_p1(self.x, self.cells, self.phi)
        ON.tag_facets_p1(self.x, self.cells, self.c2f, self.f2c, self.phi, ct)
        ON.assemble_p1(self.x, self.cells, self.c2f, self.f2c, self.phi, self.f, ct, p["active"],
                       p["slots_cells"], p["entities"], p["slots_boundary"], p["ghost"],
                       p["slots_ghost"], 1.0, self.nnz)

    def measure(self, steps, warmup, one_core=True):
        ON = self.ON
        cores = ON.num_threads()
        for _ in range(warmup):
            self.step()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.step()
        dt = (time.perf_counter() - t0) / steps
        res = {"value": self.num_cells / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "%s (%d tetrahedra), sphere level set, tags + CSR assembly (symbolic phase excluded, as for "
                         "the GPU arm), %d step(s), C/OpenMP oracle port; dolfinx/PETSc is not installable here"
                         % (self.label, self.num_cells, steps),
               "ms_per_step": dt * 1e3}
        if one_core and cores > 1:
            ON.set_num_threads(1)
            t0 = time.perf_counter()
            self.step()
            res["one_core"] = {"value": self.num_cells / (time.perf_counter() - t0), "unit": UNIT, "cores": 1}
            ON.set_num_threads(cores)
        return res


def _device_setup_for_cpu(n):
    """Config E's arrays and slot maps from the device-side symbolic phase (setup of the CPU arm when a GPU is present:
    the torch-on-CPU plumbing would take minutes at 50.9 M cells).  Nothing of this is timed."""
    import torch
    from phifem_b200 import assemble, fem, mesh_scripts, synthetic
    from phifem_b200.mesh import MeshTags
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    mesh = synthetic.box_mesh(n, device=dev)
    phi, f = synthetic.sphere_levelset(mesh.x), synthetic.ball_source(mesh.x)
    dls = mesh_scripts._DeviceLevelset(mesh, fem.Function(fem.functionspace_p1_device(mesh), phi), 1)
    ws = mesh_scripts.classify(mesh, dls)
    ents = mesh_scripts._integration_entities_dev(mesh, ws.cell_tags8, ws.facet_tags8, 4, (1, 2))
    ct, ft = MeshTags(mesh, 3, None, tags8=ws.cell_tags8), MeshTags(mesh, 2, None, tags8=ws.facet_tags8)
    plan = assemble.build_plan(mesh, ct, ft, ents, method="atomic")
    w = CpuWorkload.from_device(mesh, phi, f, plan, n)
    del mesh, plan, ws, dls
    torch.cuda.empty_cache()
    return w


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # torchrun pins OMP_NUM_THREADS=1 for its workers; the CPU arm runs on rank 0 alone and uses every
        # host core (set before libgomp is loaded)
        os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    same_config = False
    n = args.cpu_n
    try:
        import torch
        if torch.cuda.is_available() and not args.cpu_sample:
            w = _device_setup_for_cpu(args.n)       # the configuration of the GPU arm itself
            n, same_config = args.n, True
        else:
            w = CpuWorkload.from_size(n)
    except Exception as exc:                         # noqa: BLE001 -- e.g. out of host memory: fall back to the sample
        sys.stderr.write("bench.py --impl reference: full-size setup failed (%s); bounded sample n=%d\n" % (exc, n))
        w = CpuWorkload.from_size(n)
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    if same_config:          # ~0.5 s per step on 16+ threads: bound the run to about a minute
        steps, warmup = min(steps, 20), min(warmup, 2)
    res = w.measure(steps, warmup)
    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warmup, "ms_per_step": res["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": (CONFIGS["3d-p1"][1] + ", tags + strong-Dirichlet CSR assembly") % (w.num_cells, n)
                       if same_config else
                       "synthetic 3D P1 phi-FEM Poisson, Kuhn tetrahedra, sphere level set "
                       "(bounded sample n=%d of the n=%d configuration)" % (n, args.n),
                       "name": "3d-p1", "same_config_as_gpu_arm": same_config},
            "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample", "one_core") if k in res},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class Workload:
    """One problem resident on one device: mesh, level set, source, tag workspace, assembly plan, outputs.  `step()` is
    one pass of the hot path: cell tags, facet tags, assembly of the operator and the load vector."""

    def __init__(self, mesh, phi, f, args, problem=None, degree=1, ls_kw=None, cell_pass=None):
        import torch
        from phifem_b200 import assemble, fem, mesh_scripts
        from phifem_b200.mesh import MeshTags
        self.mesh, self.phi, self.f, self.problem, self.args = mesh, phi, f, problem, args
        self.torch, self.assemble_mod, self.ms = torch, assemble, mesh_scripts
        dev = mesh.device
        t0 = time.perf_counter()
        mesh.c2f  # facet topology (mesh-level symbolic, once per mesh)
        mesh.detj_bounds()
        torch.cuda.synchronize()
        self.topology_s = time.perf_counter() - t0
        self.phi_asm, self.f_asm = phi, f
        self.V = fem.functionspace_p1_device(mesh)
        fn = fem.Function(self.V, phi)
        if args.detection_degree > 1 and problem is None:
            from phifem_b200 import synthetic
            Vd = fem.functionspace(mesh, args.detection_degree)
            phi_det = synthetic.sphere_levelset(Vd.dof_coordinates_dev(), **(ls_kw or {}))
            self.dls = mesh_scripts._DeviceLevelset(mesh, fem.Function(Vd, phi_det), args.detection_degree)
        else:
            self.dls = mesh_scripts._DeviceLevelset(mesh, fn, 1)
        self.ws = mesh_scripts.TagWorkspace(mesh)
        if problem is not None:
            problem.classify(self.dls, self.ws)
        else:
            mesh_scripts.classify(mesh, self.dls, ws=self.ws)
        torch.cuda.synchronize()
        self.counters = self.ws.counters.cpu().numpy()
        t0 = time.perf_counter()
        tdim = mesh.topology.dim
        ws = self.ws
        if problem is not None:
            self.plan = problem.build_plan(ws.cell_tags8, ws.facet_tags8)
            if getattr(problem, "mode", "rows") == "exchange":
                self.plan.method, self.plan.blocked, self.plan.rowsplan = "atomic", None, None
            self.data, self.b = problem.data, problem.b_local
        else:
            ctags, ftags = MeshTags(mesh, tdim, None, tags8=ws.cell_tags8), MeshTags(mesh, tdim - 1, None,
                                                                                      tags8=ws.facet_tags8)
            ents = mesh_scripts._integration_entities_dev(mesh, ws.cell_tags8, ws.facet_tags8, 4, (1, 2))
            if degree == 2:
                # P2 trial/test space and P2 level set: phi_h / f_h = interpolants at the P2 nodes (main.py:85-90)
                from phifem_b200 import synthetic
                Vw = fem.functionspace(mesh, 2)
                Xd = Vw.dof_coordinates_dev()
                self.phi_asm = synthetic.sphere_levelset(Xd, **(ls_kw or {}))
                self.f_asm = synthetic.ball_source(Xd, **({"center": DISC_CENTER} if ls_kw else {}))
                del Xd
                self.plan = assemble.build_plan(mesh, ctags, ftags, ents, V=Vw, V_phi=Vw)
            else:
                self.plan = assemble.build_plan(mesh, ctags, ftags, ents, method=args.scatter, capacity=args.capacity,
                                                order=args.order, geometry=args.geometry,
                                                cell_pass=cell_pass or args.cell_pass,
                                                rows_per_tile=args.rows_per_tile)
            self.data, self.b = self.plan.new_outputs()
        torch.cuda.synchronize()
        self.symbolic_first_call_ms = (time.perf_counter() - t0) * 1e3
        self.symbolic_ms = self.symbolic_first_call_ms
        if problem is None and degree == 1 and getattr(self.plan, "method", "") == "rows" and not args.no_replan:
            # the first call of a process also grows the scratch pool and the allocator by several GB (driver work, paid
            # once); what a time-stepping code pays whenever the cut pattern changes is the RE-plan: timed here
            times = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                again = assemble.build_plan(mesh, ctags, ftags, ents, method=args.scatter, capacity=args.capacity,
                                            order=args.order, geometry=args.geometry,
                                            cell_pass=cell_pass or args.cell_pass, rows_per_tile=args.rows_per_tile)
                torch.cuda.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
                del again
            self.symbolic_ms = min(times)
        self.graph = None

    def step(self, events=None, split=False):
        """events: CUDA events recorded at the phase boundaries.  split=True (the untimed breakdown loop) runs the
        assembly pass by pass so that events separate its kernels."""
        k = 0

        def mark():
            nonlocal k
            if events is not None:
                events[k].record()
                k += 1
        mark()
        if self.problem is not None:   # the all-reduce of "any exterior cell" overlaps the interior-facet kernel
            self.problem.classify(self.dls, self.ws, mark=mark)
            self.problem.assemble(1.0, marks=mark if split else None)
        else:
            self.ms.classify_cells(self.mesh, self.dls, self.ws)
            mark()
            self.ms.classify_facets(self.mesh, self.dls, self.ws)
            mark()
            self.assemble_mod.assemble_into(self.plan, self.phi_asm, self.f_asm, 1.0, self.data, self.b,
                                            marks=mark if split else None)
        mark()

    def capture(self):
        """The step as ONE CUDA graph (tag kernels, the all-reduce of a sharded run, assembly kernels with their
        side-stream forks): a strong-scaled rank has ~0.3 ms of kernels per step, less than the host needs to issue
        them one by one."""
        torch = self.torch
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                self.step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.step()
        torch.cuda.synchronize()
        self.graph = g

    def run(self, events=None):
        if self.graph is not None and events is None:
            self.graph.replay()
        else:
            self.step(events)

    def kernel_launches_per_step(self):
        """Kernels of libphifem_b200.so launched by one step, COUNTED with the profiler (CUPTI) on one untimed step."""
        torch = self.torch
        try:
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                self.step()
                torch.cuda.synchronize()
            names = [e.name for e in prof.events() if getattr(e, "device_type", None) is not None
                     and "cuda" in str(e.device_type).lower()]
            import re
            ours = [m.group(0) for m in (re.search(r"\bk_\w+", n) for n in names if "phifem" in n) if m]
            if ours:
                return len(ours), sorted(set(ours))
        except Exception as exc:   # noqa: BLE001
            sys.stderr.write("bench.py: kernel count through the profiler failed (%s)\n" % exc)
        return None, None

    def counts(self):
        torch, mesh, plan = self.torch, self.mesh, self.plan
        act_v = torch.zeros(mesh.num_vertices, dtype=torch.bool, device=mesh.device)
        act_v[mesh.cells[plan.active.long()].long().reshape(-1)] = True
        c = self.counters
        return {"Nc": mesh.num_cells, "Nv": mesh.num_vertices, "Nf": mesh.num_facets, "gdim": mesh.gdim,
                "nvpc": mesh.cells.shape[1], "Na": int(plan.active.numel()), "Ng": int(plan.ghost.numel()),
                "Nv_active": int(act_v.sum()), "nnz": plan.nnz, "Nrow": plan.n_rows,
                "nd": getattr(plan, "nd", mesh.cells.shape[1]),
                "Ndof_active": int((plan.indptr[1:] > plan.indptr[:-1]).sum()),
                "Ne_ds100": int(plan.entities.shape[0]),
                "halo_entries_sent": (sum(hi - lo for lo, hi in getattr(plan, "send_ranges", []))
                                      if self.problem is not None else 0),
                "interior": int(c[0]), "cut": int(c[1]), "exterior": int(c[2])}


def timed_steps(w, steps, world, sampler=None, presteps=15, after=None):
    """EXACTLY `steps` steps bracketed by barrier + synchronize, device-timed, max over ranks; per-phase means from the
    events recorded inside the timed region (eager runs) and the assembly split from a short untimed loop.  `after()`
    runs once the timed steps and the sampler have stopped, while the outputs are still those of the last timed step."""
    import torch
    import torch.distributed as dist
    dev = w.mesh.device
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(steps)]
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    # an NVML query takes milliseconds, a step two: keep the device under the same load for a fixed number of
    # untimed steps (the same on every rank: a step holds a collective) so that the sampler has seen it, then time
    # exactly `steps` steps with the sampler still running
    for _ in range(presteps):
        w.run()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        w.run(None if w.graph is not None else evs[i])
    stop.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if sampler is not None else None
    if after is not None:
        after()
    total_ms = start.elapsed_time(stop)
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    n_split = 5
    evs2 = [[torch.cuda.Event(enable_timing=True) for _ in range(8)] for _ in range(n_split)]
    for i in range(n_split):
        w.step(evs2[i], split=True)
    torch.cuda.synchronize()
    names = ["tag_cells", "tag_facets", "zero", "assemble_cells", "assemble_boundary", "assemble_ghost", "exchange"]
    src = evs2 if w.graph is not None else None
    per = {}
    for j, nm in enumerate(["tag_cells", "tag_facets", "assembly"]):
        if src is None:
            per[nm] = statistics.mean(evs[i][j].elapsed_time(evs[i][j + 1]) for i in range(steps))
        elif nm != "assembly":
            per[nm] = statistics.mean(evs2[i][j].elapsed_time(evs2[i][j + 1]) for i in range(n_split))
        else:
            per[nm] = statistics.mean(evs2[i][2].elapsed_time(evs2[i][7]) for i in range(n_split))
    for j, nm in enumerate(names):
        if j >= 2:
            per[nm] = statistics.mean(evs2[i][j].elapsed_time(evs2[i][j + 1]) for i in range(n_split))
    if w.plan.method == "rows":
        per["assemble_surface"] = per.pop("assemble_ghost")      # ghost penalty + one-sided term, one pass
        per.pop("assemble_boundary")
    return total_ms / steps, per, clocks


DUMP_SAMPLE = 1 << 20    # entries kept of a longer output array (--dump-outputs)
DUMP_SEED = 0


def dump_outputs(w, outdir):
    """What a caller of compute_tags_measures + assemble_strong_dirichlet receives from the step just run -- cell and
    facet tags, CSR pattern and values, load vector -- as outdir/<name>.npy (tags float32, the rest float64; every value
    exact).  An array longer than DUMP_SAMPLE entries keeps DUMP_SAMPLE of them, at sorted positions drawn with DUMP_SEED
    from its length alone: two builds that compute the same arrays write the same files, 40 MB at most."""
    import torch
    os.makedirs(outdir, exist_ok=True)
    arrays = {"cell_tags": (w.ws.cell_tags8, np.float32), "facet_tags": (w.ws.facet_tags8, np.float32),
              "A_indptr": (w.plan.indptr, np.float64), "A_indices": (w.plan.indices, np.float64),
              "A_data": (w.data, np.float64), "b": (w.b, np.float64)}
    for name, (t, dtype) in arrays.items():
        t = t.reshape(-1)
        if t.numel() > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(DUMP_SEED).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t[torch.from_numpy(pos).to(t.device)]
        np.save(os.path.join(outdir, name + ".npy"), t.cpu().numpy().astype(dtype))


def roofline_of(w, per, ms_per_step, clocks):
    ab = algorithmic_bytes(w.counts())
    ab_survey = algorithmic_bytes(w.counts(), tag_bytes=4)
    plan = w.plan
    peak, peak_src = _peaks()
    dominant = max(("tag_cells", "tag_facets", "assemble_cells"), key=lambda k_: per[k_])
    # the row-gather kernel is the whole assembly (cells + ghost + one-sided terms, pattern read, CSR
    # values and b written): SURVEY.md 8(d) B_asm; the atomic cell kernel alone moves less
    asm_bytes = ab["assembly"] if plan.method in ("rows", "blocked") else ab["cells_kernel"]
    kbytes = {"tag_cells": ab["tags_cells"], "tag_facets": ab["tags_facets"], "assemble_cells": asm_bytes}[dominant]
    achieved = kbytes / (per[dominant] * 1e-3) / 1e9
    tiles = plan.rowsplan.tiles if plan.method == "rows" else None
    kernel_names = {"tag_cells": "k_tag_cells_p1", "tag_facets": "k_tag_facets",
                    "assemble_cells": {"rows": ("k_assemble_push_p1" if tiles.push is not None else "k_assemble_tiles_p1")
                                       if tiles is not None else "k_assemble_rows_p1",
                                       "blocked": "k_assemble_blocked_p1", "atomic": "k_assemble_cells_p1",
                                       "pk-atomic": "k_assemble_cells_pk"}[plan.method]}
    roofline = {"bound": "hbm", "kernel": kernel_names[dominant], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": kbytes,
                "algorithmic_bytes": "SURVEY.md 8(d) with the tag arrays at the ONE byte per entity the kernels write "
                                     "(int32 MeshTags are widened on demand outside the timed region); "
                                     "`step_frac_survey_int32_tags` keeps the survey's 4-byte yardstick for comparison "
                                     "with round 1",
                "step_bytes": ab["total"],
                "step_achieved_gbs": ab["total"] / (ms_per_step * 1e-3) / 1e9,
                "step_frac": ab["total"] / (ms_per_step * 1e-3) / 1e9 / peak,
                "step_frac_survey_int32_tags": ab_survey["total"] / (ms_per_step * 1e-3) / 1e9 / peak,
                "kernels_ms": per,
                "kernels_gbs": {"tag_cells": ab["tags_cells"] / per["tag_cells"] / 1e6,
                                "tag_facets": ab["tags_facets"] / per["tag_facets"] / 1e6,
                                "assemble_cells": asm_bytes / per["assemble_cells"] / 1e6}}
    if plan.method == "rows" and w.mesh.gdim == 3:
        # the cell pass is bound by fp64 issue, not by HBM: 146 fp64 instructions per (row, cell) record (SASS
        # count of cell_row<3>, DESIGN.md section 4) against 64 fp64 lanes per clock per SM; 85 with the cached cell
        # geometry (cell_row_geom<3>); ~200 per cell evaluation of the cell-once pass
        per_record = 200 if tiles is not None else (85 if plan.rowsplan.cell_geom is not None else 146)
        n_eval = tiles.n_cell_slots if tiles is not None else plan.rowsplan.cells.n_records
        lanes = n_eval * float(per_record)
        peak_lanes = 148 * 64 * ((clocks or {}).get("sm_max_mhz") or 1965) * 1e6
        roofline["fp64_issue"] = {"kernel": kernel_names["assemble_cells"], "fp64_instructions_per_record": per_record,
                                  "records": n_eval,
                                  "achieved_tera_lane_instr_per_s": lanes / (per["assemble_cells"] * 1e-3) / 1e12,
                                  "peak_tera_lane_instr_per_s": peak_lanes / 1e12,
                                  "frac": lanes / (per["assemble_cells"] * 1e-3) / peak_lanes}
    return roofline, ab, dominant


def scatter_info(plan):
    out = {"method": plan.method}
    if getattr(plan, "blocked", None):
        out.update({"blocks": plan.blocked.n_blocks, "capacity": plan.blocked.capacity,
                    "bin_shape": plan.blocked.bin_shape, "recompute_factor": plan.blocked.redundancy,
                    "plan_bytes": plan.blocked.index_bytes()})
    rp = getattr(plan, "rowsplan", None)
    if rp:
        out.update({"order": rp.order, "max_row_nnz": rp.max_row_nnz, "cell_pass": rp.cell_pass})
        if rp.tiles is not None:
            out.update({"rows_per_tile": rp.tiles.rows_per_tile, "tiles": rp.tiles.n_tiles, "chunks": rp.tiles.n_chunks,
                        "cell_evaluations": rp.tiles.n_cell_slots, "recompute_factor": rp.tiles.recompute})
        out.update({"rows_cells_surface": [rp.tiles.n_listed if rp.tiles is not None else rp.cells.n_listed,
                                           rp.surface.n_listed],
                    "records_cells_ghost_onesided": [rp.n_cell_records, rp.n_ghost_records, rp.n_entity_records],
                    "lane_padding": [rp.cells.padding(), rp.surface.padding()],
                    "cell_geometry": "cached per plan (64 B per active cell)" if rp.cell_geom is not None
                    else "from the vertex coordinates",
                    "plan_bytes": rp.index_bytes()})
    return out


def measure_e2e(w, args, degree):
    """Public API, pinned host buffers in, pinned host buffers out."""
    import warnings

    import torch
    from phifem_b200 import assemble, fem, mesh_scripts
    mesh, plan, dev = w.mesh, w.plan, w.mesh.device
    phi_h = w.phi.cpu().pin_memory()
    f_h = w.f_asm.cpu().pin_memory()
    phi_asm_h = w.phi_asm.cpu().pin_memory() if degree == 2 else phi_h
    out_h = {"ct": torch.empty(mesh.num_cells, dtype=torch.int8).pin_memory(),
             "ft": torch.empty(mesh.num_facets, dtype=torch.int8).pin_memory(),
             "data": torch.empty(plan.nnz, dtype=torch.float64).pin_memory(),
             "b": torch.empty(0, dtype=torch.float64)}
    # box mode keeps the rows of every vertex of the background mesh; 61 % of them (config E) are empty -- no cell of
    # Omega_h touches the vertex -- and their entry of b is a structural zero: the load vector crosses PCIe compacted to
    # the rows of the pattern (the index list is part of the plan, fetched once)
    active_rows = torch.nonzero(plan.indptr[1:] > plan.indptr[:-1]).reshape(-1)
    out_h["b"] = torch.empty(active_rows.numel(), dtype=torch.float64).pin_memory()
    rows_h = active_rows.to(torch.int32).cpu()
    bytes_in = int(phi_h.numel() * 8 + (phi_asm_h.numel() * 8 if degree == 2 else 0) + f_h.numel() * 8)
    bytes_out = int(sum(t.numel() * t.element_size() for t in out_h.values()))

    class Slot:
        """One step in flight: its streams, events, pinned output buffers and the device tensors its copies read."""

        def __init__(self, outputs):
            self.main, self.side = torch.cuda.Stream(), torch.cuda.Stream()
            self.phi_up, self.f_done, self.tags_done = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
            self.side_done, self.done = torch.cuda.Event(), torch.cuda.Event()
            self.out = outputs
            self.keep, self.pending = None, False

        def wait(self):
            if self.pending:
                self.done.synchronize()
                self.keep, self.pending = None, False

    asm_done = torch.cuda.Event()   # the plan's surface scratch is shared: the assemblies of two steps do not overlap
    asm_done.record()

    def issue(sl):
        """Queue one whole step on the slot's streams; the only host wait inside is the counter read of
        compute_tags_measures (an event of THIS slot's stream)."""
        with torch.cuda.stream(sl.main):
            # host level set -> device once; the same device-resident Function feeds the tags and (for P1) the
            # assembly, as a user holding one phi_h would write it
            phi_d = phi_h.to(dev, non_blocking=True)
            sl.phi_up.record()
            # the source term FOLLOWS the level set over PCIe (side stream, after the level set has landed: two uploads
            # at once share the link and delay the tag kernels) while the tag kernels run
            with torch.cuda.stream(sl.side):
                sl.side.wait_event(sl.phi_up)
                f_d = f_h.to(dev, non_blocking=True)
                sl.f_done.record()
            fn_h = fem.Function(w.V, phi_d)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                ct_, ft_, _, ds_, _ = mesh_scripts.compute_tags_measures(mesh, fn_h, 1, box_mode=True)
            # the tags (one byte per entity, as the kernels write them; MeshTags widens to int32 on the host)
            # leave on a side stream while the assembly runs
            sl.tags_done.record()
            with torch.cuda.stream(sl.side):
                sl.side.wait_event(sl.tags_done)
                sl.out["ct"].copy_(ct_.tags8, non_blocking=True)
                sl.out["ft"].copy_(ft_.tags8, non_blocking=True)
                sl.side_done.record()
            sl.main.wait_event(sl.f_done)
            sl.main.wait_event(asm_done)
            A_, b_ = assemble.assemble_strong_dirichlet(plan, phi_d if degree == 1 else phi_asm_h, f_d, stab_coef=1.0)
            asm_done.record()
            sl.out["data"].copy_(A_.data, non_blocking=True)
            bc = b_.index_select(0, active_rows)
            sl.out["b"].copy_(bc, non_blocking=True)
            sl.main.wait_event(sl.side_done)
            sl.done.record()
            sl.keep, sl.pending = (phi_d, f_d, ct_, ft_, A_, b_, bc, ds_), True   # alive until the copies have run

    def run(depth, steps):
        slots = [Slot(out_h)] + [Slot({k_: torch.empty_like(v).pin_memory() for k_, v in out_h.items()})
                                 for _ in range(depth - 1)]
        for k_ in range(2 * depth):
            slots[k_ % depth].wait()
            issue(slots[k_ % depth])
        for sl in slots:
            sl.wait()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k_ in range(steps):
            sl = slots[k_ % depth]
            sl.wait()               # this slot's previous step has landed in its host buffers
            issue(sl)
        for sl in slots:
            sl.wait()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / steps

    e2e_steps = max(2, min(args.steps, 5))
    dt1 = run(1, e2e_steps)
    api = ("compute_tags_measures(box_mode=True) + assemble_strong_dirichlet(plan, ...) with "
           "pinned host level set / source in and pinned host tags (1 byte per cell / facet) + CSR values "
           "+ b on the %d non-empty rows of the %d out," % (rows_h.numel(), plan.n_rows)
           + " source-term upload overlapped with the tag kernels, tag copies with the assembly; "
           "assembly plan (symbolic phase) reused; ")
    out = {"value": mesh.num_cells / dt1, "unit": UNIT, "ms_per_step": dt1 * 1e3,
           "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
           "api": api + "one step at a time", "one_step_at_a_time_ms": dt1 * 1e3}
    if not getattr(args, "no_e2e_pipeline", False):
        # two steps in flight on two streams with their own pinned output buffers: the uploads, the tag kernels and the
        # assembly of step k + 1 run under the download of step k (PCIe is full duplex, the download is the long leg)
        dt2 = run(2, 2 * e2e_steps)
        out["two_steps_in_flight_ms"] = dt2 * 1e3
        if dt2 < dt1:
            out.update({"value": mesh.num_cells / dt2, "ms_per_step": dt2 * 1e3,
                        "api": api + "TWO steps in flight (every step's copies inside the timed region, %d steps "
                                     "timed, pinned output buffers double-buffered); one step at a time: %.2f ms"
                                     % (2 * e2e_steps, dt1 * 1e3)})
    return out


def measure_e2e_dist(w, args, world):
    """The end-to-end leg of a multi-GPU run: every rank uploads the level set and the source term of ITS slab from
    pinned host memory, runs the sharded classification (with its exchange) and the assembly of its owned rows, and
    downloads its tags, owned CSR values and owned load-vector entries -- each GPU over its own PCIe link.  Time = the
    maximum over the ranks of the wall clock around K synchronised steps; value = all owned cells / that time."""
    import torch
    import torch.distributed as dist
    prob, mesh, dev = w.problem, w.mesh, w.mesh.device
    phi_h = prob.phi.cpu().pin_memory()
    f_h = prob.f.cpu().pin_memory()
    data0, b0 = prob.assemble(1.0)
    out_h = {"ct": torch.empty(mesh.num_cells, dtype=torch.int8).pin_memory(),
             "ft": torch.empty(mesh.num_facets, dtype=torch.int8).pin_memory(),
             "data": torch.empty(data0.numel(), dtype=torch.float64).pin_memory(),
             "b": torch.empty(b0.numel(), dtype=torch.float64).pin_memory()}
    upload = torch.cuda.Stream()
    f_done, phi_up = torch.cuda.Event(), torch.cuda.Event()

    class Slot:
        """Host buffers of one step in flight, device staging copies of its results (the problem's own tag / value
        arrays are rewritten by the next step while this step's download is still running), its copy stream."""

        def __init__(self, outputs, staged):
            self.out, self.copy, self.staged = outputs, torch.cuda.Stream(), staged
            self.dev = ({k_: torch.empty(v.shape, dtype=v.dtype, device=dev) for k_, v in outputs.items()}
                        if staged else None)
            self.tags_done, self.asm_done, self.done = torch.cuda.Event(), torch.cuda.Event(), torch.cuda.Event()
            self.pending = False

        def wait(self):
            if self.pending:
                self.done.synchronize()
                self.pending = False

    def issue(sl):
        main = torch.cuda.current_stream()
        prob.phi.copy_(phi_h, non_blocking=True)      # (the classifier and the plan read these device arrays in place)
        phi_up.record()
        with torch.cuda.stream(upload):
            upload.wait_event(phi_up)
            prob.f.copy_(f_h, non_blocking=True)
            f_done.record()
        prob.classify(w.dls, w.ws)
        ct, ft = w.ws.cell_tags8, w.ws.facet_tags8
        if sl.staged:
            sl.dev["ct"].copy_(ct, non_blocking=True)
            sl.dev["ft"].copy_(ft, non_blocking=True)
            ct, ft = sl.dev["ct"], sl.dev["ft"]
        sl.tags_done.record()
        with torch.cuda.stream(sl.copy):
            sl.copy.wait_event(sl.tags_done)
            sl.out["ct"].copy_(ct, non_blocking=True)
            sl.out["ft"].copy_(ft, non_blocking=True)
        main.wait_event(f_done)
        data, b = prob.assemble(1.0)
        if sl.staged:
            sl.dev["data"].copy_(data, non_blocking=True)
            sl.dev["b"].copy_(b, non_blocking=True)
            data, b = sl.dev["data"], sl.dev["b"]
        sl.asm_done.record()
        with torch.cuda.stream(sl.copy):
            sl.copy.wait_event(sl.asm_done)
            sl.out["data"].copy_(data, non_blocking=True)
            sl.out["b"].copy_(b, non_blocking=True)
            sl.done.record()
        if not sl.staged:
            main.wait_event(sl.done)      # one step at a time: the next step rewrites the arrays being downloaded
        sl.pending = True

    def run(depth, nsteps):
        slots = [Slot(out_h, depth > 1)] + [Slot({k_: torch.empty_like(v).pin_memory() for k_, v in out_h.items()}, True)
                                            for _ in range(depth - 1)]
        for k_ in range(2 * depth):
            slots[k_ % depth].wait()
            issue(slots[k_ % depth])
        for sl in slots:
            sl.wait()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k_ in range(nsteps):
            sl = slots[k_ % depth]
            sl.wait()
            issue(sl)
        for sl in slots:
            sl.wait()
        torch.cuda.synchronize()
        t = torch.tensor([(time.perf_counter() - t0) / nsteps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    steps = max(2, min(args.steps, 5))
    dt1 = run(1, steps)
    dt2 = None if getattr(args, "no_e2e_pipeline", False) else run(2, 2 * steps)
    dt = dt1 if dt2 is None or dt1 <= dt2 else dt2
    cells = torch.tensor([prob.n_owned_cells], dtype=torch.int64, device=dev)
    h2d = torch.tensor([phi_h.numel() * 8 + f_h.numel() * 8], dtype=torch.int64, device=dev)
    d2h = torch.tensor([sum(t.numel() * t.element_size() for t in out_h.values())], dtype=torch.int64, device=dev)
    for t in (cells, h2d, d2h):
        dist.all_reduce(t)
    out = {"value": int(cells.item()) / dt, "unit": UNIT, "ms_per_step": dt * 1e3,
           "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": int(d2h.item()),
           "one_step_at_a_time_ms": dt1 * 1e3,
           "api": "per rank: pinned host level set / source of its slab in, SlabProblem.classify (sharded tags with "
                  "their exchange) + SlabProblem.assemble (owned rows), pinned host tags (1 byte per local cell / "
                  "facet) + owned CSR values + owned b out; every GPU over its own PCIe link; max over the %d ranks, "
                  "bytes summed over the ranks; %s" % (world, "one step at a time" if dt is dt1 else
                                                       "TWO steps in flight (results staged in a second device buffer, "
                                                       "pinned output buffers double-buffered, every step's copies "
                                                       "inside the timed region)")}
    if dt2 is not None:
        out["two_steps_in_flight_ms"] = dt2 * 1e3
    return out


def time_to_solution(w):
    """SURVEY.md 8(f-3): tags + assembly + the solve that follows them in the demos (reference
    demo/strong-dirichlet/flower/main.py:138-157 hands the system to MUMPS), here Jacobi-BiCGStab on the CSR operator
    in HBM.  One run, wall clock with synchronisation on both sides."""
    import torch
    from phifem_b200 import solve
    from phifem_b200.assemble import CSRMatrix
    A = CSRMatrix(w.plan.indptr, w.plan.indices, w.data, (w.plan.n_rows, w.plan.n_rows))
    # ten untimed iterations first: the first solve of a process grows the allocator by ~1 GB of vectors and column ids
    # (0.2-0.6 s of driver work on a process that already holds the benchmark's arrays); a time-stepping code pays it once
    solve.bicgstab(A, w.b, rtol=1e-8, maxiter=10)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    w.step()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    x, info = solve.bicgstab(A, w.b, rtol=1e-8, maxiter=4000)
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return {"total_ms": (t2 - t0) * 1e3, "tags_and_assembly_ms": (t1 - t0) * 1e3, "solve_ms": (t2 - t1) * 1e3,
            "solver": "Jacobi-BiCGStab, rtol 1e-8, fused iteration on the active rows (phifem_b200/solve.py, "
                      "csrc/solve.cu phifem_bicgstab_iterate); warm process (ten untimed iterations first)",
            "iterations": info.iterations, "residual": info.residual, "converged": bool(info.converged),
            "unknowns": info.n_active}


def multi_gpu_parity(dev, rank, world, n=12, peer=True):
    """A small problem through the SAME sharded code path (scatter from rank 0, sharded tags with the all-reduce,
    owner-computes assembly), merged on rank 0 and compared BITWISE with rank 0's single-GPU operator."""
    import torch
    import torch.distributed as dist
    from phifem_b200 import assemble, fem, mesh_scripts, partition, synthetic
    from phifem_b200.mesh import MeshTags
    ref = None
    gmesh = gphi = gf = None
    if rank == 0:
        gmesh = synthetic.box_mesh(n, device=dev)
        gphi = synthetic.sphere_levelset(gmesh.x, radius=0.37)
        gf = torch.from_numpy(np.random.default_rng(7).uniform(-1, 1, gmesh.num_vertices)).to(dev)
        dls = mesh_scripts._DeviceLevelset(gmesh, fem.Function(fem.functionspace_p1_device(gmesh), gphi), 1)
        ws = mesh_scripts.classify(gmesh, dls)
        ents = mesh_scripts._integration_entities_dev(gmesh, ws.cell_tags8, ws.facet_tags8, 4, (1, 2))
        plan = assemble.build_plan(gmesh, MeshTags(gmesh, 3, None, tags8=ws.cell_tags8),
                                   MeshTags(gmesh, 2, None, tags8=ws.facet_tags8), ents)
        data, b = plan.new_outputs()
        assemble.assemble_into(plan, gphi, gf, 1.0, data, b)
        ref = (plan.indptr.cpu().numpy(), plan.indices.cpu().numpy(), data.cpu().numpy(), b.cpu().numpy(),
               ws.cell_tags8.cpu().numpy())
    prob = partition.PartitionedProblem.scatter(gmesh, gphi, gf, rank, world, device=dev)
    if peer:
        prob.enable_peer_flags()
    dls = mesh_scripts._DeviceLevelset(prob.mesh, fem.Function(fem.functionspace_p1_device(prob.mesh), prob.phi), 1)
    ws = mesh_scripts.TagWorkspace(prob.mesh)
    prob.classify(dls, ws)
    prob.build_plan(ws.cell_tags8, ws.facet_tags8)
    prob.assemble(1.0)
    rows, indptr, cols, data, b = (t.cpu().numpy() for t in prob.owned_csr())
    mine = (rows, indptr, cols, data, b, prob.global_cell[prob.cell_owned].cpu().numpy(),
            ws.cell_tags8[prob.cell_owned].cpu().numpy())
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    ok = None
    if rank == 0:
        ip, ix, dd, bb, ct = ref
        seen = np.zeros(len(bb), dtype=np.int64)
        seen_c = np.zeros(len(ct), dtype=np.int64)
        ok = True
        for rows, indptr, cols, data, b, cells_owned, tags in parts:
            seen[rows] += 1
            seen_c[cells_owned] += 1
            ok &= bool(np.array_equal(tags, ct[cells_owned]))
            ok &= bool(np.array_equal(np.diff(indptr), ip[rows + 1] - ip[rows]))
            if not ok:
                break
            sl = np.concatenate([np.arange(ip[r], ip[r + 1]) for r in rows]) if len(rows) else np.zeros(0, dtype=np.int64)
            ok &= bool(np.array_equal(cols, ix[sl]) and np.array_equal(data, dd[sl]) and np.array_equal(b, bb[rows]))
        ok &= bool(np.all(seen == 1) and np.all(seen_c == 1))
    flag = torch.tensor([1 if (ok or ok is None) else 0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item())


def strong_scaling(args, dev, rank, world):
    """Config E itself -- ONE 6 n^3-tetrahedra mesh -- cut along the Morton curve into `world` ranges of equal WEIGHT
    (exterior 1, interior 3, cut 10: SURVEY.md 8e), partition computed once on rank 0 and scattered; every rank
    classifies its share (redundant halo included) and assembles the rows it owns; the step is one CUDA graph."""
    import torch
    import torch.distributed as dist
    from phifem_b200 import partition, synthetic
    t0 = time.perf_counter()
    gmesh = gphi = gf = weights = None
    n_cells = 6 * args.n ** 3
    if rank == 0:
        gmesh = synthetic.box_mesh(args.n, device=dev)
        gphi, gf = synthetic.sphere_levelset(gmesh.x), synthetic.ball_source(gmesh.x)
        neg = (gphi < 0)[gmesh.cells.long()]
        inside, outside = neg.all(dim=1), (~neg).all(dim=1)
        weights = torch.where(inside, 3.0, torch.where(outside, 1.0, 10.0)).to(torch.float64)
        del neg, inside, outside
    prob = partition.PartitionedProblem.scatter(gmesh, gphi, gf, rank, world, weights=weights, device=dev)
    peer = (not args.no_peer) and prob.enable_peer_flags()
    del gmesh, gphi, gf, weights
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    scatter_s = time.perf_counter() - t0
    w = Workload(prob.mesh, prob.phi, prob.f, args, problem=prob)
    graph = False
    if not args.no_graph:
        try:
            w.capture()
            graph = True
        except Exception as exc:   # noqa: BLE001
            sys.stderr.write("bench.py: CUDA-graph capture of the sharded step failed (%s); eager launches\n" % exc)
            w.graph = None
    graph_all = torch.tensor([1 if graph else 0], device=dev)
    dist.all_reduce(graph_all, op=dist.ReduceOp.MIN)
    if not bool(graph_all.item()):
        w.graph, graph = None, False
    ms, per, _ = timed_steps(w, args.steps, world, presteps=5)
    stats = torch.tensor([prob.mesh.num_cells, prob.n_owned_cells, w.symbolic_ms, w.topology_s * 1e3,
                          per["tag_cells"] + per["tag_facets"], per["assembly"]], dtype=torch.float64, device=dev)
    allst = [torch.empty_like(stats) for _ in range(world)]
    dist.all_gather(allst, stats)
    allst = torch.stack(allst).cpu().numpy()
    owned_total = int(allst[:, 1].sum())
    assert owned_total == n_cells, "the ranks' owned cells do not partition the mesh"
    return {"n_gpus": world, "cells_total": n_cells, "ms_per_step": ms, "value": n_cells / (ms * 1e-3), "unit": UNIT,
            "cuda_graph": graph, "scatter_s": scatter_s,
            "exchange": "exterior-cell counts stored into the peers' HBM over NVLink (csrc/peer.cu)" if peer else
                        "8-byte NCCL all-reduce",
            "partition": "Morton curve of the cell centroids, ranges of equal weight (exterior 1 / interior 3 / cut 10), "
                         "computed once on rank 0 and scattered; rows owned by the lowest rank touching them; "
                         "redundantly classified halo (cells sharing a vertex with a cell touching an owned row); one "
                         "8-byte all-reduce per step, no halo exchange",
            "local_cells": [int(v) for v in allst[:, 0]], "owned_cells": [int(v) for v in allst[:, 1]],
            "symbolic_ms_max": float(allst[:, 2].max()), "topology_ms_max": float(allst[:, 3].max()),
            "tags_ms": [float(v) for v in allst[:, 4]], "assembly_ms": [float(v) for v in allst[:, 5]]}


def other_config(name, args, dev, clocks):
    """Device-resident step of another BASELINE.json configuration (same metric, same timing rules, fewer keys)."""
    import copy

    import torch
    from phifem_b200 import synthetic
    n = CONFIGS[name][0]
    a = copy.copy(args)
    a.config, a.n, a.no_replan = name, n, True
    ls_kw = {}
    if name.startswith("2d"):
        mesh = synthetic.rectangle_mesh(n, device=dev)
        ls_kw.update(center=DISC_CENTER, radius=DISC_RADIUS)
    else:
        mesh = synthetic.box_mesh(n, device=dev)
    phi = synthetic.sphere_levelset(mesh.x, **ls_kw)
    f = synthetic.ball_source(mesh.x, **({"center": DISC_CENTER} if ls_kw else {}))
    w = Workload(mesh, phi, f, a, degree=2 if name.endswith("p2") else 1, ls_kw=ls_kw)
    for _ in range(a.warmup):
        w.step()
    torch.cuda.synchronize()
    ms, per, _ = timed_steps(w, a.steps, 1, presteps=3)
    roof, ab, dominant = roofline_of(w, per, ms, clocks)
    c = w.counts()
    return {"workload": CONFIGS[name][1] % (mesh.num_cells, n), "cells": mesh.num_cells, "ms_per_step": ms,
            "value": mesh.num_cells / (ms * 1e-3), "unit": UNIT, "kernels_ms": per, "step_frac": roof["step_frac"],
            "dominant_kernel": roof["kernel"], "dominant_frac": roof["frac"],
            "counts": {k: v for k, v in c.items() if k in ("interior", "cut", "exterior", "nnz", "Na", "Ng",
                                                           "Ndof_active")},
            "method": w.plan.method}


def _bind_to_gpu_cores(index):
    """One process per GPU: run on the host cores NVML lists as local to this GPU, so that the pinned buffers of the
    end-to-end leg are first touched on the memory node the GPU's PCIe root hangs off (on a two-socket host the copies of
    the ranks bound to the far socket otherwise cross the inter-socket link).  A no-op where the mask does not narrow the
    process's own (single-node hosts and VMs)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        words = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index), 16)
        local = {64 * i + b for i, w_ in enumerate(words) for b in range(64) if (int(w_) >> b) & 1}
        mine = os.sched_getaffinity(0)
        if local & mine and (local & mine) != mine:
            os.sched_setaffinity(0, local & mine)
            sys.stderr.write("bench.py: rank on GPU %d bound to host cores %s\n" % (index, sorted(local & mine)))
    except Exception as exc:   # noqa: BLE001
        sys.stderr.write("bench.py: no GPU-local core binding (%s)\n" % exc)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from phifem_b200 import synthetic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        _bind_to_gpu_cores(local_rank)

    n = args.n
    degree = 2 if args.config.endswith("p2") else 1
    ls_kw = {}
    reorder_ms = None
    problem = None

    def make_mesh(kind):
        nonlocal reorder_ms
        if args.config.startswith("2d"):
            mesh = synthetic.rectangle_mesh(n, device=dev)
            ls_kw.update(center=DISC_CENTER, radius=DISC_RADIUS)
        else:
            mesh = synthetic.box_mesh(n, device=dev)
        if kind == "unstructured":
            # SURVEY.md 8(d): vertex jitter +-0.2 h (seed 0), random cell permutation (seed 1), random vertex
            # relabelling (seed 2); then -- as part of the mesh-level symbolic phase, like dolfinx's own reordering at
            # mesh creation -- renumbered along the Morton curve.  Level set and source are interpolated on THAT mesh.
            mesh = synthetic.unstructured_variant_device(mesh, jitter=0.2, seed=0)
            torch.cuda.synchronize()
            t_re = time.perf_counter()
            if not args.no_reorder:
                mesh = mesh.reordered(args.curve)
            torch.cuda.synchronize()
            reorder_ms = (time.perf_counter() - t_re) * 1e3
        phi = synthetic.sphere_levelset(mesh.x, **ls_kw)
        f = synthetic.ball_source(mesh.x, **({"center": DISC_CENTER} if ls_kw else {}))
        return mesh, phi, f

    parity_ok = strong = None
    if world > 1:
        from phifem_b200 import dist as pdist
        if not args.no_parity:
            parity_ok = multi_gpu_parity(dev, rank, world, peer=not args.no_peer)
        if args.scaling == "strong" or not args.no_strong:
            strong = strong_scaling(args, dev, rank, world)
            torch.cuda.empty_cache()
        problem = pdist.SlabProblem(n, rank, world, dev, mode=args.dist_mode)
        if not args.no_peer:
            problem.enable_peer_flags()
        mesh, phi, f = problem.mesh, problem.phi, problem.f
    else:
        mesh, phi, f = make_mesh(args.mesh)
    w = Workload(mesh, phi, f, args, problem=problem, degree=degree, ls_kw=ls_kw)
    plan = w.plan
    peer_halo = (problem is not None and args.dist_mode == "exchange" and not args.no_peer
                 and problem.enable_peer_halo())
    _sym = (w.symbolic_ms, w.topology_s, w.symbolic_first_call_ms, getattr(plan, "symbolic", None))

    for _ in range(args.warmup):
        w.step()
    torch.cuda.synchronize()
    dump = (lambda: dump_outputs(w, args.dump_outputs)) if args.dump_outputs else None
    ms_per_step, per, clocks = timed_steps(w, args.steps, world, sampler=ClockSampler(local_rank), after=dump)

    n_cells_local = problem.n_owned_cells if problem is not None else mesh.num_cells
    n_cells_total = n_cells_local
    if world > 1:
        t = torch.tensor([n_cells_local], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        n_cells_total = int(t.item())
    value = n_cells_total / (ms_per_step * 1e-3)
    counts = w.counts()
    roofline, ab, dominant = roofline_of(w, per, ms_per_step, clocks)
    traffic_file = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_file) and args.config == "3d-p1" and n == CONFIGS["3d-p1"][0] and world == 1 \
            and args.mesh == "structured" and plan.method == "rows" and plan.rowsplan.tiles is None:
        with open(traffic_file) as fh:
            tr = json.load(fh)
        roofline["traffic"] = tr.get(dominant)
        roofline["traffic_source"] = tr.get("source", "profiles/traffic.json (ncu --set full capture of this command)")
    launches, launch_names = w.kernel_launches_per_step()
    plan_check_ms = None
    if world == 1 and hasattr(plan, "matches"):
        # what a moving-interface loop pays after every re-tag to learn whether the plan can be reused
        from phifem_b200.mesh import MeshTags
        tdim = mesh.topology.dim
        tags_now = (MeshTags(mesh, tdim, None, tags8=w.ws.cell_tags8), MeshTags(mesh, tdim - 1, None, tags8=w.ws.facet_tags8))
        assert plan.matches(*tags_now), "the plan of the timed steps is not the plan of their tags"
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plan.matches(*tags_now)
        plan_check_ms = (time.perf_counter() - t0) * 1e3

    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(w, args, degree) if world == 1 else measure_e2e_dist(w, args, world)
    tts = None
    if world == 1 and degree == 1 and not args.no_solve and plan.method == "rows":
        try:
            tts = time_to_solution(w)
        except Exception as exc:   # noqa: BLE001
            tts = {"error": str(exc)}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and args.config == "3d-p1" and args.mesh == "structured":
        if args.cpu_sample or plan.method != "rows":
            cpu = CpuWorkload.from_size(args.cpu_n).measure(3, 1)
        else:       # the configuration itself: arrays and slot maps of the plan just timed, copied to the host
            cpu = CpuWorkload.from_device(mesh, phi, f, plan, n).measure(3, 1)
        cpu.pop("ms_per_step")

    # ---- the unstructured variant of the same configuration (VERDICT round 1, row "star") ----------------------
    unstructured = None
    if world == 1 and args.config == "3d-p1" and args.mesh == "structured" and not args.no_unstructured:
        structured_ms = ms_per_step
        del w
        torch.cuda.empty_cache()
        try:
            umesh, uphi, uf = make_mesh("unstructured")
            uw = Workload(umesh, uphi, uf, args)
            for _ in range(args.warmup):
                uw.step()
            ums, uper, _ = timed_steps(uw, args.steps, 1, presteps=3)
            uroof, _, _ = roofline_of(uw, uper, ums, clocks)
            unstructured = {"mesh": "SURVEY.md 8(d) variant of the same configuration: vertex jitter +-0.2 h (seed 0), "
                                    "cells permuted (seed 1), vertices relabelled (seed 2), then renumbered "
                                    + ("along the Morton curve" if getattr(umesh, "reorder_curve", "") == "morton" else
                                       "in count-balanced pencils (slabs of equal vertex count along x, pencils of equal "
                                       "count along y, sorted along z: parameter-free; chosen by curve=auto for meshes "
                                       "with grid connectivity, the Morton curve otherwise)")
                                    + " (Mesh.reordered, timed as reorder_ms); level set and source "
                                    "interpolated on that mesh",
                            "curve": getattr(umesh, "reorder_curve", args.curve),
                            "cells": umesh.num_cells, "ms_per_step": ums, "value": umesh.num_cells / (ums * 1e-3),
                            "unit": UNIT, "ratio_to_structured": ums / structured_ms,
                            "step_frac": uroof["step_frac"], "kernels_ms": uper, "reorder_ms": reorder_ms,
                            "symbolic_ms": uw.symbolic_ms, "topology_s": uw.topology_s,
                            "counts": {k: v for k, v in uw.counts().items() if k in ("interior", "cut", "exterior",
                                                                                    "nnz", "Na", "Ng")}}
            del uw, umesh, uphi, uf
        except Exception as exc:   # noqa: BLE001
            unstructured = {"error": str(exc)}
        torch.cuda.empty_cache()
        w = None

    # ---- the other configurations of BASELINE.json (VERDICT round 1, item 8): one short measurement each --------
    others = None
    if world == 1 and args.config == "3d-p1" and args.mesh == "structured" and not args.no_others:
        w = None
        torch.cuda.empty_cache()
        others = {}
        for name in ("2d-p1", "2d-p2", "3d-p2"):
            try:
                others[name] = other_config(name, args, dev, clocks)
            except Exception as exc:   # noqa: BLE001
                others[name] = {"error": str(exc)}
            torch.cuda.empty_cache()

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": (CONFIGS[args.config][1] + "%s, tags + strong-Dirichlet CSR assembly")
                                       % (n_cells_local, n, " per unit cube joined by a thin tube across the "
                                          "partition boundaries" if world > 1 else ""),
                           "name": args.config, "mesh": args.mesh + (
                               "" if args.mesh == "structured" else
                               (": jitter 0.2 h, cells permuted, vertices relabelled" +
                                (", NOT renumbered" if args.no_reorder else
                                 ", renumbered (Mesh.reordered, curve=%s)" % args.curve))),
                           "cells_total": n_cells_total, "counts": counts,
                           "l2_policy": "inputs larger than L2 (%.1f GB streamed per step)"
                                        % (ab["total"] / 1e9),
                           "partition": ("single GPU" if world == 1 else
                                         "1 slab of the global box per rank, owned CSR rows, "
                                         + ("owner computes its rows from 2 redundantly classified ghost "
                                            "layers: one 8-byte all-reduce per step, no halo exchange"
                                            if args.dist_mode == "rows" else
                                            ("halo contributions pushed into the owners' HBM over NVLink and added "
                                             "there by the same kernel (phifem_halo_exchange)" if peer_halo else
                                             "NCCL halo exchange (grouped send / recv + index_add_)"))
                                         + ("; the 8 bytes travel as stores into the peers' HBM over NVLink (csrc/peer.cu)"
                                            if getattr(problem, "peer", None) is not None else "")),
                           "tags_dtype": "int8 on the device (int32 MeshTags.values widened on demand)",
                           "timed": "tag kernels + zeroing + assembly kernels; symbolic phase excluded; "
                                    "kernels_ms: tag_* and assembly from events inside the timed region, "
                                    "the assemble_* split from an untimed pass-by-pass loop"},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": clocks,
                "gpu_launches": (launches if launches is not None else
                                 {"rows": 7, "blocked": 5, "atomic": 7, "pk-atomic": 9}[plan.method]) * args.steps,
                "gpu_launches_per_step": launches, "gpu_kernels": launch_names,
                "gpu_launches_source": "counted with the CUPTI profiler on one untimed step" if launches is not None
                else "table (profiler unavailable)",
                "symbolic_ms": _sym[0], "topology_s": _sym[1], "symbolic_first_call_ms": _sym[2],
                "symbolic": {"builder": _sym[3], "symbolic_ms": "re-plan (pattern + row lists) on a warm process, best of "
                             "2; symbolic_first_call_ms also grows the allocator / scratch pool by several GB"},
                "cold_step_ms": _sym[0] + ms_per_step,
                "plan_check_ms": plan_check_ms,
                "reorder_ms": reorder_ms if args.mesh == "unstructured" else None,
                "scatter": scatter_info(plan)}
        if unstructured is not None:
            line["unstructured"] = unstructured
        if tts is not None:
            line["time_to_solution_ms"] = tts
        if others is not None:
            line["other_configs"] = others
        if world > 1:
            line["parity_ok"] = parity_ok
            line["parity"] = ("n=12 problem through PartitionedProblem.scatter + sharded tags + owner-computes assembly on "
                              "%d ranks, merged owned rows BITWISE equal to rank 0's single-GPU operator" % world)
            if strong is not None:
                line["strong"] = strong
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_JSON_FD = None


def _quiet_stdout():
    """Library chatter (e.g. "NCCL version ..." from libnccl) must not share stdout with the ONE JSON line:
    fd 1 is pointed at stderr for the run and the line is written to the saved descriptor."""
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    payload = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(payload.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_JSON_FD, payload)


def parser():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="3d-p1", choices=sorted(CONFIGS),
                    help="workload; the default is the configuration BASELINE.json's metric is quoted on")
    ap.add_argument("--n", type=int, default=None,
                    help="cells per edge (6 n^3 tetrahedra per GPU / 2 n^2 triangles); default per config")
    ap.add_argument("--cpu-n", type=int, default=80, help="size of the bounded CPU sample")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scatter", default="rows", choices=["rows", "blocked", "atomic"],
                    help="assembly strategy (row-gather / owner-computes blocks / fp64 reductions)")
    ap.add_argument("--capacity", type=int, default=None, help="contributions per block (blocked scatter)")
    ap.add_argument("--mesh", default="structured", choices=["structured", "unstructured"],
                    help="unstructured = SURVEY.md 8(d)'s variant (jitter, cell permutation, vertex relabelling), "
                         "renumbered along the Morton curve in the mesh-level symbolic phase")
    ap.add_argument("--no-reorder", action="store_true", help="unstructured mesh left in its random numbering")
    ap.add_argument("--curve", default="auto", choices=["auto", "morton", "pencil"],
                    help="renumbering of the unstructured mesh (Mesh.reordered): Morton curve / count-balanced pencils / "
                         "auto = pencils when the mesh has the connectivity of a grid")
    ap.add_argument("--no-others", action="store_true",
                    help="skip the short measurements of the other BASELINE.json configurations (2d-p1, 2d-p2, 3d-p2)")
    ap.add_argument("--no-e2e-pipeline", action="store_true",
                    help="end-to-end leg: one step at a time only (default: also two steps in flight, the faster "
                         "of the two is e2e.value, both are reported)")
    ap.add_argument("--cell-pass", default="rows", choices=["rows", "tiles", "push"],
                    help="row-gather cell pass / cell-once tile pass (csrc/assemble_tiles.cu)")
    ap.add_argument("--rows-per-tile", type=int, default=256, choices=[128, 256])
    ap.add_argument("--order", default="auto", choices=["auto", "natural", "morton"],
                    help="row processing order of the row-gather assembly")
    ap.add_argument("--geometry", action="store_true",
                    help="row-gather cell pass from a per-plan geometry table instead of the vertex coordinates "
                         "(measured slower: profiles/round2_a_geometry_kernel.md)")
    ap.add_argument("--dist-mode", default="rows", choices=["rows", "exchange"],
                    help="multi-GPU numeric strategy: owner-computes rows / per-entity kernels + halo exchange")
    ap.add_argument("--detection-degree", type=int, default=1, choices=[1, 2],
                    help="degree of the detection level set and of the detection rule (1 = the demos' setting)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--cpu-sample", action="store_true",
                    help="CPU arm on the bounded n = --cpu-n sample instead of the configuration itself")
    ap.add_argument("--no-unstructured", action="store_true", help="skip the unstructured variant (extra key)")
    ap.add_argument("--no-solve", action="store_true", help="skip time_to_solution_ms (extra key)")
    ap.add_argument("--no-replan", action="store_true", help="skip the warm re-plan timing (symbolic_ms = first call)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="multi-GPU: the headline value is always the weak-scaling slab problem; the strong-scaling "
                         "run of config E through the Morton partitioner is reported under the key `strong`")
    ap.add_argument("--no-strong", action="store_true", help="multi-GPU: skip the strong-scaling run")
    ap.add_argument("--no-parity", action="store_true", help="multi-GPU: skip the parity check (parity_ok)")
    ap.add_argument("--no-peer", action="store_true",
                    help="multi-GPU: exchange the exterior-cell counts with an NCCL all-reduce instead of peer memory")
    ap.add_argument("--no-graph", action="store_true", help="strong scaling: eager launches instead of one CUDA graph")
    ap.add_argument("--no-e2e", action="store_true", help="skip the end-to-end leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the tags, CSR arrays and load vector of the last one as DIR/<name>.npy "
                         "(one GPU, --impl ours; arrays over %d entries as a fixed seeded sample)" % DUMP_SAMPLE)
    return ap


def main():
    # the benchmark reads the tree and never writes to it (the tree may be read-only): no bytecode caches there either
    sys.dont_write_bytecode = True
    ap = parser()
    args = ap.parse_args()
    if args.n is None:
        args.n = CONFIGS[args.config][0]
    multi_gpu = args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1
    if args.config != "3d-p1" and multi_gpu:
        raise SystemExit("bench.py: the multi-GPU path runs the 3d-p1 configuration")
    if args.steps < 1:
        raise SystemExit("bench.py: --steps must be at least 1")
    if args.dump_outputs and (multi_gpu or args.impl != "ours"):
        raise SystemExit("bench.py: --dump-outputs writes the outputs of the single-GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    _quiet_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
