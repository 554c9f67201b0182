"""GPU parity against fixtures produced by the reference's OWN tools (tests/golden/make_golden.py): the rebuilt C++ tools must write
byte-identical .cdf / .cdm / .bmp files, and the C-ABI kernels must reproduce the reference class's interpolate / shape functions
bit for bit.  This pins K3 (density map) and the facade's reduceField to reference output, not only to the restated oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, bits_equal
from oracle_api import ref_check
from test_oracle_golden import read_cdf
from test_oracle_reference_tools import split_inputs

pytestmark = pytest.mark.gpu
BIN = os.path.join(ROOT, "build", "bin")


def _tool(name):
    p = os.path.join(BIN, name)
    if not os.path.exists(p):
        pytest.skip(f"{p} not built (make cpp)")
    return p


def _same(a, b):
    return open(a, "rb").read() == open(b, "rb").read()


def test_generate_sdf_files_byte_identical(tmp_path):
    exe = _tool("GenerateSDF")
    obj = os.path.join(GOLDEN, "sphere.obj")
    out = str(tmp_path / "a.cdf")
    assert subprocess.run([exe, "-r", "10 10 10", "-d", "-2 -2 -2 2 2 2", "-o", out, obj], capture_output=True).returncode == 0
    assert _same(out, os.path.join(GOLDEN, "ref_sphere.cdf"))
    out = str(tmp_path / "b.cdf")
    assert subprocess.run([exe, "-i", "-r", "4 6 5", "-o", out, obj], capture_output=True).returncode == 0
    assert _same(out, os.path.join(GOLDEN, "ref_sphere_inverted_padded.cdf"))


@pytest.mark.parametrize("mesh,args,fixture", [("bunny.obj", ["-r", "12 12 12"], "ref_bunny_12.cdf"),
                                               ("dragon.obj", ["-i", "-r", "10 10 10"], "ref_dragon_10_inverted.cdf"),
                                               ("happy_buddha.obj", ["-r", "8 8 8"], "ref_buddha_8.cdf")])
def test_generate_sdf_on_reference_meshes_byte_identical(tmp_path, mesh, args, fixture):
    """the reference's own meshes (BASELINE configs 2 / 3; happy_buddha is not watertight) through the rebuilt tool vs the reference
    tool's own output (small grids to keep the fixtures small)"""
    from conftest import ref_resource
    exe = _tool("GenerateSDF")
    obj = ref_resource(mesh)
    if obj is None:
        pytest.skip(f"{mesh} not staged (oracle/_ref/resources)")
    out = str(tmp_path / "m.cdf")
    assert subprocess.run([exe] + args + ["-o", out, obj], capture_output=True).returncode == 0
    assert _same(out, os.path.join(GOLDEN, fixture))


def test_generate_density_map_files_byte_identical(tmp_path):
    exe = _tool("GenerateDensityMap")
    src = os.path.join(GOLDEN, "ref_sphere.cdf")
    out = str(tmp_path / "nr.cdm")
    r = subprocess.run([exe, "-s", "0.15", "-r", "1000", "--no-reduction", "-o", out, src], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert _same(out, os.path.join(GOLDEN, "ref_sphere_noreduction.cdm"))            # K3, all nodes, bit for bit
    out = str(tmp_path / "red.cdm")
    r = subprocess.run([exe, "-s", "0.15", "-r", "1000", "-o", out, src], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert _same(out, os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))                # + predicate + both reduceField passes (node order, cell map)


def _bmp_equal(a, b):
    """pixel data, dimensions and format identical.  Two header fields of the reference file are not reproducible: its file-size
    field holds sizeof(BMPINFO) = 40 and SizeImage is written before it is assigned (bmp_file.cpp:76-96: uninitialised stack bytes)."""
    ra, rb = open(a, "rb").read(), open(b, "rb").read()
    return len(ra) == len(rb) and ra[:2] == rb[:2] and ra[10:34] == rb[10:34] and ra[38:54] == rb[38:54] and ra[54:] == rb[54:]


def test_bitmap_pixels_identical(tmp_path):
    exe = _tool("DiscreteFieldToBitmap")
    out = str(tmp_path / "a.bmp")
    assert subprocess.run([exe, "-s", "64", "-p", "xz", "-d", "0.25", "-o", out, os.path.join(GOLDEN, "box.cdf")], capture_output=True).returncode == 0
    assert _bmp_equal(out, os.path.join(GOLDEN, "ref_box_xz.bmp"))
    out = str(tmp_path / "b.bmp")
    assert subprocess.run([exe, "-s", "48", "-p", "yx", "-f", "1", "-c", "rs", "-o", out, os.path.join(GOLDEN, "ref_sphere_noreduction.cdm")],
                          capture_output=True).returncode == 0
    assert _bmp_equal(out, os.path.join(GOLDEN, "ref_sphere_density_yx.bmp"))


@pytest.mark.parametrize("tag,path,field", [("box", "box.cdf", 0), ("red", "ref_sphere_reduced.cdm", 0), ("red", "ref_sphere_reduced.cdm", 1),
                                            ("nr", "ref_sphere_noreduction.cdm", 1)])
def test_interpolate_kernel_matches_reference_class(dg, tag, path, field):
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = dg.CubicLagrangeDiscreteGrid(os.path.join(GOLDEN, path))
    x = q[tag + "_x"]
    phi, grad = g.interpolate(field, x, gradient=True)
    assert bits_equal(phi, q[f"{tag}_f{field}_phi"]) and bits_equal(grad, q[f"{tag}_f{field}_grad"])
    assert bits_equal(g.interpolate(field, x), q[f"{tag}_f{field}_phi_only"])


def test_shape_function_kernel_matches_reference_class(dg):
    from discregrid_b200 import _capi as capi
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = read_cdf(os.path.join(GOLDEN, "box.cdf"))
    ok = q["box_split_ok"].astype(bool)
    _c0, xi, _mi = split_inputs(g, q["box_x"][:1500][ok])
    xi = np.ascontiguousarray(xi)
    N = np.empty((len(xi), 32)); dN = np.empty((len(xi), 32, 3))
    capi.check(capi.lib.dg_shape_functions(capi.ptr(xi, capi.F64P), len(xi), capi.ptr(N, capi.F64P), capi.ptr(dN, capi.F64P)))
    assert ref_check("ref_grid_queries/box_split_N_dN", (N, dN), None, nan_equal=False)


def test_python_reduce_field_then_interpolate(dg):
    """Python mirror of reduceField (node positions from the GPU, dg_reduce_field on the host): ref_sphere.cdf reduced with the tool's
    SDF predicate must equal field 0 of the reference tool's reduced file, and the sparsified field must interpolate like it"""
    h = 0.15
    g = dg.CubicLagrangeDiscreteGrid(os.path.join(GOLDEN, "ref_sphere.cdf"))
    red = read_cdf(os.path.join(GOLDEN, "ref_sphere_reduced.cdm"))
    cs = g.cellSize()
    cell_diag = np.sqrt((cs[0] ** 2 + cs[1] ** 2) + cs[2] ** 2)
    seen = {}

    def pred(x, v):
        seen["x"] = x
        return (-6.0 * h < v + cell_diag) & (v - cell_diag < 2.0 * h)
    g.reduceField(0, pred)
    assert seen["x"].shape == (len(read_cdf(os.path.join(GOLDEN, "ref_sphere.cdf"))["nodes"][0]), 3)
    assert bits_equal(g.m_nodes[0], red["nodes"][0]) and np.array_equal(g.m_cells[0], red["cells"][0]) and np.array_equal(g.m_cell_map[0], red["cmap"][0])
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    phi, grad = g.interpolate(0, q["red_x"], gradient=True)
    assert bits_equal(phi, q["red_f0_phi"]) and bits_equal(grad, q["red_f0_grad"])
