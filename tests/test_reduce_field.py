"""SURVEY 8(f) N3 -- reduceField (cubic_lagrange_discrete_grid.cpp:1065-1174) through the C-ABI's dg_reduce_field, without a GPU:
the reference's GenerateDensityMap wrote tests/golden/ref_sphere_reduced.cdm by running both of its reduceField passes
(cmd/generate_density_map/main.cpp:137-144); the same inputs and predicates must give the same node order, cells and cell map."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, bits_equal
from test_oracle_golden import read_cdf

DBL_MAX = np.finfo(np.float64).max
H, RHO0 = 0.15, 1000.0                                   # make_golden.py: GenerateDensityMap -s 0.15 -r 1000


HOST = 2                                                 # DG_REDUCE_HOST_PASSES: this file runs without a GPU (the GPU passes: tests/test_gpu_reduce_field.py)


def reduce_field(dg, g, nodes, keep, cells, flags=0):
    from discregrid_b200 import _capi as capi
    flags |= HOST
    desc = dg.grid_desc(g["mn"], g["mx"], g["res"], g["cell"], g["inv"])
    nodes = np.ascontiguousarray(nodes, np.float64).copy(); cells = np.ascontiguousarray(cells, np.uint32).copy()
    keep = np.ascontiguousarray(keep, np.uint8)
    cmap = np.full(int(np.prod(g["res"].astype(np.uint64))), 12345, np.uint32)
    n_nodes, n_cells = C.c_uint64(), C.c_uint64()
    tm = np.zeros(5)
    capi.check(capi.lib.dg_reduce_field(C.byref(desc), capi.ptr(nodes, capi.F64P), len(nodes), keep.ctypes.data_as(C.POINTER(C.c_uint8)),
                                        capi.ptr(cells, capi.U32P), len(cells), capi.ptr(cmap, capi.U32P), flags, C.byref(n_nodes), C.byref(n_cells),
                                        capi.ptr(tm, capi.F64P)))
    reduce_field.last_timings = tm
    return nodes[:n_nodes.value], cells[:n_cells.value], cmap


def sdf_keep(g, v):
    cell_diag = np.sqrt((g["cell"][0] ** 2 + g["cell"][1] ** 2) + g["cell"][2] ** 2)          # cellSize().norm(), main.cpp:117
    return (-6.0 * H < v + cell_diag) & (v - cell_diag < 2.0 * H) & (v != DBL_MAX)                # main.cpp:137-140 and :1073


@pytest.mark.parametrize("flags", [0, 1])
def test_sdf_field_reduced_like_the_reference_tool(dg, flags):
    full = read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))
    red = read_cdf(os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))
    v = full["nodes"][0]
    nodes, cells, cmap = reduce_field(dg, full, v, sdf_keep(full, v), full["cells"][0], flags)
    assert 0 < len(nodes) < len(v) and 0 < len(cells) < len(full["cells"][0])
    assert bits_equal(nodes, red["nodes"][0])
    assert np.array_equal(cells, red["cells"][0]) and np.array_equal(cmap, red["cmap"][0])


@pytest.mark.parametrize("flags", [0, 1])
def test_density_field_reduced_like_the_reference_tool(dg, orc, flags):
    full = read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))
    red = read_cdf(os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))
    gd, res = orc.grid_desc(full["mn"], full["mx"], full["res"], full["cell"], full["inv"])
    rho = orc.density_map(gd, res, full["nodes"][0], H, RHO0, False, 0, len(full["nodes"][0]))   # what the tool sampled (pinned elsewhere)
    keep = (0.0 <= rho) & (rho <= 3.0 * RHO0) & (rho != DBL_MAX)                                 # main.cpp:141-144
    nodes, cells, cmap = reduce_field(dg, full, rho, keep, full["cells"][0], flags)
    assert bits_equal(nodes, red["nodes"][1])
    assert np.array_equal(cells, red["cells"][1]) and np.array_equal(cmap, red["cmap"][1])


def test_reduce_field_edge_cases(dg):
    from discregrid_b200 import _capi as capi
    full = read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))
    v, cells = full["nodes"][0], full["cells"][0]
    # nothing kept: empty field, every cell removed
    nodes, c, cmap = reduce_field(dg, full, v, np.zeros(len(v), np.uint8), cells)
    assert len(nodes) == 0 and len(c) == 0 and (cmap == 0xFFFFFFFF).all()
    # everything kept: all cells stay in place, nodes are only re-ordered along the Z curve; interpolation data is a permutation
    nodes, c, cmap = reduce_field(dg, full, v, np.ones(len(v), np.uint8), cells)
    assert len(nodes) == len(v) and np.array_equal(cmap, np.arange(len(cells), dtype=np.uint32))
    assert bits_equal(nodes[c], v[cells])                                                        # every cell still sees its 32 values
    assert bits_equal(np.sort(nodes), np.sort(v))
    # a field that is not in the grid's own numbering is refused (its node positions would be meaningless)
    desc = dg.grid_desc(full["mn"], full["mx"], full["res"], full["cell"], full["inv"])
    n1, n2 = C.c_uint64(), C.c_uint64()
    short = v[:100].copy(); keep = np.ones(100, np.uint8); cm = np.zeros(1000, np.uint32); cc = cells[:1].copy()
    rc = capi.lib.dg_reduce_field(C.byref(desc), capi.ptr(short, capi.F64P), 100, keep.ctypes.data_as(C.POINTER(C.c_uint8)), capi.ptr(cc, capi.U32P), 1,
                                  capi.ptr(cm, capi.U32P), 0, C.byref(n1), C.byref(n2), None)
    assert rc == capi.DG_ERR_INVALID and b"already reduced" in capi.lib.dg_last_error()


def test_tied_morton_keys_follow_the_reference_sort(dg):
    """anisotropic grid (tests/golden/make_reduce_golden.py): surviving nodes share Morton keys, so the node order is the one the
    reference's std::sort leaves -- dg_reduce_field must notice the ties by itself and reproduce it"""
    src = read_cdf(os.path.join(GOLDEN, "ref_aniso_field.cdf"))
    want = read_cdf(os.path.join(GOLDEN, "ref_aniso_reduced.cdf"))
    v = src["nodes"][0]
    keep = (0.3 <= v) & (v <= 0.9) & (v != DBL_MAX)
    nodes, cells, cmap = reduce_field(dg, src, v, keep, src["cells"][0])
    assert reduce_field.last_timings[4] == 1.0                                                   # the tie path was taken
    assert bits_equal(nodes, want["nodes"][0]) and np.array_equal(cells, want["cells"][0]) and np.array_equal(cmap, want["cmap"][0])


def test_facade_reduce_field_glue_without_gpu(dg, tmp_path):
    """the C++ facade's reduceField (predicate loop + dg_reduce_field + resize) on both fields of a .cdm, node positions interposed
    by the oracle (tests/cpp/reduce_facade_check.cpp): field 0 must be the reference tool's reduced field 0"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "build", "bin", "reduce_facade_check")
    if not os.path.exists(exe):
        pytest.skip("build/bin/reduce_facade_check not built (make cpp)")
    src_path = os.path.join(GOLDEN, "ref_sphere_noreduction.cdm")
    out = str(tmp_path / "red.cdm")
    r = subprocess.run([exe, src_path, str(H), str(RHO0), out], capture_output=True, text=True, env=dict(os.environ, DG_REDUCE_FIELD_HOST="1"))
    assert r.returncode == 0, r.stdout + r.stderr
    got, src, red = read_cdf(out), read_cdf(src_path), read_cdf(os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))
    assert bits_equal(got["nodes"][0], red["nodes"][0]) and np.array_equal(got["cells"][0], red["cells"][0]) and np.array_equal(got["cmap"][0], red["cmap"][0])
    v1 = src["nodes"][1]
    n1, c1, m1 = reduce_field(dg, src, v1, (0.0 <= v1) & (v1 <= 3.0 * RHO0) & (v1 != DBL_MAX), src["cells"][1])
    assert bits_equal(got["nodes"][1], n1) and np.array_equal(got["cells"][1], c1) and np.array_equal(got["cmap"][1], m1)


@pytest.mark.parametrize("mn,mx,res,lo,hi", [([-1, -1, -1], [1, 1, 1], (16, 16, 16), 0.5, 0.7), ([-1, -2, -1], [1, 1, 3], (20, 9, 14), 0.5, 1.2),
                                             ([0, 0, 0], [1, 2, 4], (5, 7, 3), 0.0, 5.0), ([-1, -1, -1], [1, 1, 1], (40, 40, 40), 0.55, 0.7)])
def test_against_the_reference_library(dg, orc, tmp_path, mn, mx, res, lo, hi):
    """random blob fields reduced by dg_reduce_field and by the reference class (its results stored as digests, oracle_api.ref_check)"""
    from oracle_api import RefGrid, ref_check
    import sys
    sys.path.insert(0, GOLDEN)
    from make_reduce_golden import synthetic_field, write_cdf
    gd, r, v, cells = synthetic_field(orc, mn, mx, res, 7)
    src = str(tmp_path / "in.cdf")
    write_cdf(src, mn, mx, res, gd[6:9], gd[9:12], v, cells, np.arange(len(cells), dtype=np.uint32))

    def reference():
        ref = RefGrid(src); ref.reduce_window(0, lo, hi); ref.save(str(tmp_path / "out.cdf")); ref.close()
        want = read_cdf(str(tmp_path / "out.cdf"))
        return want["nodes"][0], want["cells"][0], want["cmap"][0]
    g = dict(mn=np.array(mn, float), mx=np.array(mx, float), res=np.array(res, np.uint32), cell=gd[6:9], inv=gd[9:12])
    nodes, c2, cmap = reduce_field(dg, g, v, (lo <= v) & (v <= hi) & (v != DBL_MAX), cells)
    assert ref_check(f"reduce_field/{mn}/{mx}/{res}/{lo}/{hi}", (nodes, c2, cmap), reference, nan_equal=False)


def test_threaded_sort_replay_equals_std_sort():
    """tests/cpp/sort_replay_check.cpp: the tie path's multithreaded replay of libstdc++'s introsort leaves records with equal keys
    exactly where std::sort leaves them (random ties, few keys, presorted, adversarial input that exhausts the depth budget)"""
    import subprocess
    from conftest import ROOT
    exe = os.path.join(ROOT, "build", "bin", "sort_replay_check")
    if not os.path.exists(exe):
        pytest.skip("build/bin/sort_replay_check not built (make cpp)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and r.stdout.strip().endswith("OK"), r.stdout + r.stderr
