"""CPU-only: the bench line the driver parses.  The argument parser's defaults, the byte yardstick of SURVEY.md 8(d) as
`bench.algorithmic_bytes` states it, and the committed lines of the final build (profiles/round2_r4x_bench_default.json,
round2_r4z_bench_reference.json, round2_r4s_scale_8.json): every key of the contract present, the numbers consistent
with each other (value = cells / time, roofline fractions = achieved / peak, end-to-end bytes > 0 and slower than the
device-resident step, clocks at their maximum without a throttle reason)."""
import json
import os

import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(name):
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        pytest.skip(name + " not committed")
    with open(path) as fh:
        return json.load(fh)


def test_defaults_of_the_command_line():
    a = bench.parser().parse_args([])
    assert a.gpus == 1 and a.impl == "ours" and a.config == "3d-p1" and a.warmup >= 3 and a.steps >= 10
    assert a.cell_pass == "rows" and not a.no_e2e and not a.no_e2e_pipeline and not a.no_others
    assert a.dump_outputs is None
    assert bench.CONFIGS["3d-p1"][0] == 204          # 6 * 204^3 = 50 937 984 tetrahedra: BASELINE.json configs[4]
    assert 6 * 204 ** 3 == 50937984


def test_dump_outputs_writes_exact_values_and_a_seeded_sample(tmp_path):
    """--dump-outputs on a stand-in workload of host tensors: one .npy per output, values exact in float32 / float64,
    short arrays whole, long ones sampled at the same positions on every call, under 64 MB in all."""
    import types

    import numpy as np
    import torch
    n_long = bench.DUMP_SAMPLE + 12345
    rng = np.random.default_rng(5)
    plan = types.SimpleNamespace(indptr=torch.arange(0, 3 * 1001, 3, dtype=torch.int32),
                                 indices=torch.from_numpy(rng.integers(0, 2 ** 31 - 1, n_long).astype(np.int32)))
    ws = types.SimpleNamespace(cell_tags8=torch.from_numpy(rng.integers(1, 4, n_long).astype(np.int8)),
                               facet_tags8=torch.from_numpy(rng.integers(0, 5, 777).astype(np.int8)))
    w = types.SimpleNamespace(ws=ws, plan=plan, data=torch.from_numpy(rng.standard_normal(n_long)),
                              b=torch.from_numpy(rng.standard_normal(1000)))
    bench.dump_outputs(w, str(tmp_path / "a"))
    bench.dump_outputs(w, str(tmp_path / "b"))
    names = {"cell_tags", "facet_tags", "A_indptr", "A_indices", "A_data", "b"}
    assert {p.stem for p in (tmp_path / "a").iterdir()} == names
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 * 2 ** 20
    got = {nm: np.load(tmp_path / "a" / (nm + ".npy")) for nm in names}
    for nm in names:
        assert np.array_equal(got[nm], np.load(tmp_path / "b" / (nm + ".npy")))
    assert got["cell_tags"].dtype == got["facet_tags"].dtype == np.float32
    assert got["A_data"].dtype == got["A_indices"].dtype == got["A_indptr"].dtype == got["b"].dtype == np.float64
    assert np.array_equal(got["facet_tags"], ws.facet_tags8.numpy()) and np.array_equal(got["b"], w.b.numpy())
    assert np.array_equal(got["A_indptr"], plan.indptr.numpy())
    pos = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(n_long, bench.DUMP_SAMPLE, replace=False))
    assert np.array_equal(got["A_data"], w.data.numpy()[pos])
    assert np.array_equal(got["A_indices"], plan.indices.numpy()[pos])
    assert np.array_equal(got["cell_tags"], ws.cell_tags8.numpy()[pos])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--dump-outputs", "out", "--impl", "reference"],
                                  ["--dump-outputs", "out", "--gpus", "2"]])
def test_bench_refuses_arguments_it_cannot_honour(argv, monkeypatch):
    monkeypatch.setattr("sys.argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit, match="bench.py: "):
        bench.main()


def test_algorithmic_bytes_is_the_yardstick_of_the_survey():
    c = _line("round2_r4x_bench_default.json")["config"]["counts"]
    ab1, ab4 = bench.algorithmic_bytes(c, tag_bytes=1), bench.algorithmic_bytes(c, tag_bytes=4)
    nc, nv, nf, na, nnz, nrow = c["Nc"], c["Nv"], c["Nf"], c["Na"], c["nnz"], c["Nrow"]
    # SURVEY.md 8(d): B_tags = 4 nvpc Nc + 8 Ndof_phi + 4 Nc + 4 nfpc Nc + 4 Nf with int32 tags
    assert ab4["tags_cells"] + ab4["tags_facets"] == 4 * 4 * nc + 8 * nv + 4 * nc + 4 * 4 * nc + 4 * nf
    assert ab1["tags_cells"] + ab1["tags_facets"] == 4 * 4 * nc + 8 * nv + nc + 4 * 4 * nc + nf
    nva = c["Nv_active"]
    assert ab4["assembly"] == (4 * 4 * na + 8 * 3 * nva + 8 * nva + 8 * nva + 4 * na + 8 * c["Ng"] + 12 * nnz
                               + 4 * (nrow + 1) + 8 * nrow)
    assert ab1["total"] == ab1["tags_cells"] + ab1["tags_facets"] + ab1["assembly"] < ab4["total"]


def test_committed_default_line_keeps_the_contract():
    d = _line("round2_r4x_bench_default.json")
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "clocks", "gpu_launches"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["unit"] == "cells/s"
    cfg = d["config"]
    assert "workload" in cfg and "model" not in cfg and cfg["cells_total"] == 50937984
    assert "larger than L2" in cfg["l2_policy"]
    assert d["value"] == pytest.approx(cfg["cells_total"] / (d["ms_per_step"] * 1e-3), rel=1e-9)
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and r["kernel"] == "k_assemble_rows_p1"
    assert r["frac"] == pytest.approx(r["achieved"] / r["peak"], rel=1e-9) and 0.0 < r["frac"] < 1.0
    assert r["achieved"] == pytest.approx(r["algorithmic_bytes_per_launch"] / (r["kernels_ms"]["assemble_cells"] * 1e-3) / 1e9,
                                          rel=1e-9)
    assert r["step_bytes"] == bench.algorithmic_bytes(cfg["counts"])["total"]
    assert r["step_frac"] == pytest.approx(r["step_bytes"] / (d["ms_per_step"] * 1e-3) / 1e9 / r["peak"], rel=1e-9)
    # DRAM traffic of the dominant kernel (ncu) does not exceed its algorithmic bytes: no wasted re-reads
    assert 0 < r["traffic"] <= r["algorithmic_bytes_per_launch"]
    k = r["kernels_ms"]
    assert k["tag_cells"] + k["tag_facets"] + k["assembly"] == pytest.approx(d["ms_per_step"], rel=0.03)
    cpu = d["cpu_baseline"]
    assert cpu["kind"] == "port" and cpu["cores"] >= 1 and cpu["unit"] == "cells/s" and 0 < cpu["value"] < d["value"]
    assert "n=204" in cpu["sample"]
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["unit"] == "cells/s"
    assert e["value"] < d["value"] and e["value"] == pytest.approx(cfg["cells_total"] / (e["ms_per_step"] * 1e-3), rel=1e-9)
    assert e["ms_per_step"] == pytest.approx(min(e["one_step_at_a_time_ms"], e["two_steps_in_flight_ms"]), rel=1e-9)
    # PCIe cannot have moved the bytes faster than a Gen5 x16 link does
    assert e["d2h_bytes_per_step"] / (e["ms_per_step"] * 1e-3) < 64e9
    c = d["clocks"]
    assert c["sm_mhz"] == c["sm_max_mhz"] and not [x for x in c["reasons"] if "slowdown" in x or "thermal" in x]
    assert d["gpu_launches"] == d["gpu_launches_per_step"] * d["steps"] > 0 and len(d["gpu_kernels"]) >= 5
    assert d["plan_check_ms"] < d["ms_per_step"] and d["cold_step_ms"] == pytest.approx(d["symbolic_ms"] + d["ms_per_step"])
    u = d["unstructured"]
    assert u["cells"] == cfg["cells_total"] and u["ratio_to_structured"] <= 1.3       # VERDICT round 1, row "star"
    assert set(d["other_configs"]) == {"2d-p1", "2d-p2", "3d-p2"}
    for v in d["other_configs"].values():
        assert v["value"] == pytest.approx(v["cells"] / (v["ms_per_step"] * 1e-3), rel=1e-9)
    assert d["time_to_solution_ms"]["total_ms"] > d["ms_per_step"]


def test_committed_reference_arm_line():
    d = _line("round2_r4z_bench_reference.json")
    ours = _line("round2_r4x_bench_default.json")
    assert d["impl"] == "reference" and d["metric"] == ours["metric"] and d["unit"] == ours["unit"]
    assert d["higher_is_better"] is True and d["config"]["workload"] == ours["config"]["workload"]
    assert d["config"]["same_config_as_gpu_arm"] is True and d["config"]["name"] == ours["config"]["name"]
    assert d["value"] == pytest.approx(ours["config"]["cells_total"] / (d["ms_per_step"] * 1e-3), rel=1e-9)
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_committed_eight_gpu_line():
    d = _line("round2_r4s_scale_8.json")
    one = _line("round2_r4x_bench_default.json")
    assert d["n_gpus"] == 8 and d["scaling"] == "weak" and d["parity_ok"] is True
    assert d["config"]["cells_total"] == 8 * one["config"]["cells_total"]
    assert d["value"] == pytest.approx(d["config"]["cells_total"] / (d["ms_per_step"] * 1e-3), rel=1e-9)
    assert d["value"] / (8 * one["value"]) > 0.9                      # weak-scaling efficiency
    s = d["strong"]
    assert s["cells_total"] == one["config"]["cells_total"] and s["n_gpus"] == 8
    assert one["ms_per_step"] / (8 * s["ms_per_step"]) > 0.7          # strong-scaling efficiency (VERDICT round 1, item 4)
