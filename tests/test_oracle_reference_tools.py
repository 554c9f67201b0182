"""Pins the oracle's GRID half (node positions, connectivity, interpolate, shape functions, density map) -- without a GPU -- to
fixtures produced by the reference's own tools and grid class: the UNMODIFIED reference sources compiled against the Eigen
stand-in oracle/ref_eigen (tests/golden/make_golden.py; that build reproduces box.cdf byte for byte before anything is generated).
Caveat stated in DESIGN.md: the stand-in fixes Eigen's 3-term norm() order ((a0+a1)+a2), which real Eigen could not confirm here."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, bits_equal
from oracle_api import ref_check
from test_oracle_golden import read_cdf, read_obj

DBL_MAX = np.finfo(np.float64).max


def _grid(orc, g):
    return orc.grid_desc(g["mn"], g["mx"], g["res"], g["cell"], g["inv"])


def test_generate_sdf_custom_domain(orc):
    g = read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))                  # GenerateSDF -r "10 10 10" -d "-2 -2 -2 2 2 2" sphere.obj
    V, F = read_obj(os.path.join(GOLDEN, "sphere.obj"))
    assert np.array_equal(g["mn"], [-2, -2, -2]) and np.array_equal(g["mx"], [2, 2, 2]) and list(g["res"]) == [10, 10, 10]
    gd, res = orc.grid_desc(g["mn"], g["mx"], g["res"])
    assert bits_equal(gd[6:9], g["cell"]) and bits_equal(gd[9:12], g["inv"])
    assert bits_equal(orc.mesh(V, F).sample_sdf(gd, res), g["nodes"][0])
    assert np.array_equal(orc.build_cells(res), g["cells"][0])


def test_generate_sdf_inverted_padded_anisotropic(orc):
    g = read_cdf(os.path.join(GOLDEN, "ref_sphere_inverted_padded.cdf"))  # GenerateSDF -i -r "4 6 5" sphere.obj
    V, F = read_obj(os.path.join(GOLDEN, "sphere.obj"))
    mn, mx = orc.generate_sdf_domain(V)
    assert bits_equal(mn, g["mn"]) and bits_equal(mx, g["mx"])
    gd, res = orc.grid_desc(mn, mx, g["res"])
    assert bits_equal(orc.mesh(V, F).sample_sdf(gd, res, sign=-1.0), g["nodes"][0])
    assert np.array_equal(orc.build_cells(res), g["cells"][0])


def test_density_map_no_reduction_bit_exact(orc):
    g = read_cdf(os.path.join(GOLDEN, "ref_sphere_noreduction.cdm"))      # GenerateDensityMap -s 0.15 -r 1000 --no-reduction
    assert g["n_fields"] == 2
    gd, res = _grid(orc, g)
    want = g["nodes"][1]
    got = orc.density_map(gd, res, g["nodes"][0], 0.15, 1000.0, True, 0, len(want))
    assert bits_equal(got, want)
    assert (want == 0).any() and (want > 0).any()


def test_density_map_predicate_matches_reduced_file(orc):
    """with reduction the tool samples with the predicate (DBL_MAX where rejected) and then sparsifies: every surviving node value
    of field 1 must be a value the oracle computes with the predicate on, and the counts must be consistent"""
    full = read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))
    red = read_cdf(os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))
    gd, res = _grid(orc, full)
    mine = orc.density_map(gd, res, full["nodes"][0], 0.15, 1000.0, False, 0, len(full["nodes"][0]))
    assert (mine == DBL_MAX).any()
    assert set(np.unique(red["nodes"][1]).tolist()) <= set(np.unique(mine).tolist())
    assert len(red["cells"][1]) < len(full["cells"][0]) and (red["cmap"][1] == 0xFFFFFFFF).any()


@pytest.mark.parametrize("tag,path,field", [("box", "box.cdf", 0), ("red", "ref_sphere_reduced.cdm", 0), ("red", "ref_sphere_reduced.cdm", 1),
                                            ("nr", "ref_sphere_noreduction.cdm", 1)])
def test_interpolate_matches_reference_class(orc, tag, path, field):
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = read_cdf(os.path.join(GOLDEN, path))
    gd, res = _grid(orc, g)
    x = q[tag + "_x"]
    phi, grad = orc.interpolate(gd, res, g["nodes"][field], x, grad=True, cells=g["cells"][field], cell_map=g["cmap"][field])
    assert bits_equal(phi, q[f"{tag}_f{field}_phi"]) and bits_equal(grad, q[f"{tag}_f{field}_grad"])
    assert bits_equal(orc.interpolate(gd, res, g["nodes"][field], x, grad=False, cells=g["cells"][field], cell_map=g["cmap"][field])[0],
                      q[f"{tag}_f{field}_phi_only"])
    assert (phi == DBL_MAX).any() and (phi != DBL_MAX).any()


def split_inputs(g, x):
    """xi = c0*x - c1 for in-domain points, with the reference's operations (cubic_lagrange_discrete_grid.cpp:909-928), in numpy"""
    mi = ((x - g["mn"]) * g["inv"]).astype(np.uint32)
    mi = np.minimum(mi, g["res"] - 1)
    lo = g["mn"] + mi.astype(np.float64) * g["cell"]
    hi = lo + g["cell"]
    denom = hi - lo
    c0 = 2.0 / denom
    c1 = (hi + lo) / denom
    return c0, c0 * x - c1, mi


def test_split_api_matches_reference_class(orc):
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = read_cdf(os.path.join(GOLDEN, "box.cdf"))
    x = q["box_x"][:1500]
    ok = q["box_split_ok"].astype(bool)
    inside = np.all((g["mn"] <= x) & (x <= g["mx"]), axis=1)
    assert np.array_equal(ok, inside)
    c0, xi, mi = split_inputs(g, x[ok])
    assert bits_equal(c0, q["box_split_c0"][ok])
    N, dN = orc.shape_functions(xi)
    assert ref_check("ref_grid_queries/box_split_N_dN", (N, dN), None, nan_equal=False)       # shape_function_ pinned to the reference's code
    cell_id = g["res"][1] * g["res"][0] * mi[:, 2] + g["res"][0] * mi[:, 1] + mi[:, 0]
    assert np.array_equal(g["cells"][0][cell_id], q["box_split_cell"][ok])
    assert bits_equal(q["box_split_phi"][ok], q["box_f0_phi"][:1500][ok]) and bits_equal(q["box_split_grad"][ok], q["box_f0_grad"][:1500][ok])


REAL_MESH_FIXTURES = [("bunny.obj", "ref_bunny_12.cdf", 1.0), ("dragon.obj", "ref_dragon_10_inverted.cdf", -1.0), ("happy_buddha.obj", "ref_buddha_8.cdf", 1.0)]


@pytest.mark.parametrize("mesh,fixture,sign", REAL_MESH_FIXTURES)
def test_real_meshes_through_reference_tool(orc, mesh, fixture, sign):
    """the reference GenerateSDF on its own meshes (bunny 12^3; dragon 10^3 --invert; happy_buddha 8^3: 855k triangles, not watertight):
    the oracle reproduces the files' coefficients (meshes from oracle/_ref/resources)"""
    from conftest import ref_resource
    path = ref_resource(mesh)
    if path is None:
        pytest.skip(f"{mesh} not staged")
    g = read_cdf(os.path.join(GOLDEN, fixture))
    V, F = read_obj(path)
    mn, mx = orc.generate_sdf_domain(V)
    assert bits_equal(mn, g["mn"]) and bits_equal(mx, g["mx"])          # non-cubic bounding box: padding arithmetic incl. the norm order of the stand-in
    gd, res = orc.grid_desc(mn, mx, g["res"])
    assert bits_equal(orc.mesh(V, F).sample_sdf(gd, res, sign=sign), g["nodes"][0])


def test_oracle_equals_the_references_real_addfunction(orc):
    """refg_add_function_sdf drives the reference's own CubicLagrangeDiscreteGrid::addFunction with the GenerateSDF functor
    (cubic_lagrange_discrete_grid.cpp:780-899; cmd/generate_sdf/main.cpp:92-105): node coefficients, connectivity table and node count
    equal the oracle's restatement bit for bit -- also inverted and on an anisotropic resolution (the reference's results stored as
    digests, oracle_api.ref_check)"""
    from oracle_api import RefAddFunction
    import discregrid_b200 as dg
    t = dg.bumpy_torus(30, 24, 1.0, 0.4, 0.05, 7, 5)
    mesh = orc.mesh(t.vertices, t.faces)
    mn, mx = orc.generate_sdf_domain(t.vertices)
    for res, invert in (((9, 7, 5), False), ((6, 6, 6), True)):
        gd, r = orc.grid_desc(mn, mx, res)
        want = mesh.sample_sdf(gd, r, sign=-1.0 if invert else 1.0)
        reference = lambda: RefAddFunction(t.vertices, t.faces).add_function(mn, mx, res, invert=invert, want_nodes=True, want_cells=True)[1:]
        assert ref_check(f"ref_add_function/torus30x24/{res}/invert={invert}", (want, orc.build_cells(r)), reference, nan_equal=False)
