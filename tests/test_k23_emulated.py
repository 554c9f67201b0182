"""The product's K2 (pack / interpolate / shape functions) and K3 (density map) device code and launchers, compiled for the CPU by
tests/emu and compared bit for bit with the reference class's own results (tests/golden/ref_grid_queries.npz, .cdm files written by the
reference tools) and with the oracle -- the CPU-suite counterpart of tests/test_gpu_k2_interp.py / test_gpu_k3_density.py /
test_gpu_reference_tools.py.  The TMA staging of K2 is replaced by a plain copy in the emulation; everything else is the kernel's code."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, bits_equal
from oracle_api import ref_check
from test_oracle_golden import read_cdf
from test_oracle_reference_tools import split_inputs

LIBS = [os.path.join(ROOT, "build", "bin", "libk23emu.so"), os.path.join(ROOT, "build", "bin", "libk23emu_knobs.so")]      # default; K3_FAST_DIV
_dp, _u32p = C.POINTER(C.c_double), C.POINTER(C.c_uint32)
DBL_MAX = np.finfo(np.float64).max


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


class Emu:
    def __init__(self, so):
        if not os.path.exists(so):
            pytest.skip(f"{so} not built (make cpp)")
        self.lib = C.CDLL(so)
        self.lib.emu_field_create.restype = C.c_void_p
        self.lib.emu_field_create.argtypes = [_dp, _u32p, _dp, _u32p, C.c_uint64, _u32p]
        self.lib.emu_field_destroy.argtypes = [C.c_void_p]
        self.lib.emu_interpolate.argtypes = [C.c_void_p, _dp, C.c_uint64, _dp, _dp]
        self.lib.emu_shape_functions.argtypes = [_dp, C.c_uint64, _dp, _dp]
        self.lib.emu_density_map.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_uint64, C.c_uint64, _dp]

    def field(self, orc, g, f, closed_form=False):
        gd, res = orc.grid_desc(g["mn"], g["mx"], g["res"], g["cell"], g["inv"])
        nodes = np.ascontiguousarray(g["nodes"][f], np.float64)
        cells = None if closed_form else np.ascontiguousarray(g["cells"][f], np.uint32)
        cmap = None if closed_form else np.ascontiguousarray(g["cmap"][f], np.uint32)
        h = self.lib.emu_field_create(_p(gd, _dp), _p(res, _u32p), _p(nodes, _dp), _p(cells, _u32p), len(g["cells"][f]), _p(cmap, _u32p))
        assert h
        return h, (gd, res, nodes, cells, cmap)          # keep the arrays alive


@pytest.fixture(scope="module", params=LIBS, ids=[os.path.basename(p) for p in LIBS])
def emu(request):
    return Emu(request.param)


@pytest.mark.parametrize("tag,path,field,closed", [("box", "box.cdf", 0, False), ("box", "box.cdf", 0, True), ("red", "ref_sphere_reduced.cdm", 0, False),
                                                   ("red", "ref_sphere_reduced.cdm", 1, False), ("nr", "ref_sphere_noreduction.cdm", 1, False)])
def test_emulated_interpolate_matches_reference_class(emu, orc, tag, path, field, closed):
    """value + gradient and value-only, plain / reduced fields, explicit and closed-form connectivity, out-of-domain and removed cells"""
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = read_cdf(os.path.join(GOLDEN, path))
    h, keep = emu.field(orc, g, field, closed)
    x = np.ascontiguousarray(q[tag + "_x"]); n = len(x)
    phi = np.zeros(n); grad = np.full((n, 3), np.nan)
    assert emu.lib.emu_interpolate(h, _p(x, _dp), n, _p(phi, _dp), _p(grad, _dp)) == 0
    assert bits_equal(phi, q[f"{tag}_f{field}_phi"]) and bits_equal(grad, q[f"{tag}_f{field}_grad"])
    phi2 = np.zeros(n)
    assert emu.lib.emu_interpolate(h, _p(x, _dp), n, _p(phi2, _dp), None) == 0
    assert bits_equal(phi2, q[f"{tag}_f{field}_phi_only"])
    assert (phi == DBL_MAX).any() and (phi != DBL_MAX).any()
    # a query count that is not a multiple of the warp / block size
    m = 77
    assert emu.lib.emu_interpolate(h, _p(x, _dp), m, _p(phi2, _dp), None) == 0 and bits_equal(phi2[:m], phi[:m])
    emu.lib.emu_field_destroy(h)


def test_emulated_shape_functions_match_reference_class(emu):
    q = np.load(os.path.join(GOLDEN, "ref_grid_queries.npz"))
    g = read_cdf(os.path.join(GOLDEN, "box.cdf"))
    ok = q["box_split_ok"].astype(bool)
    _c0, xi, _mi = split_inputs(g, q["box_x"][:1500][ok])
    xi = np.ascontiguousarray(xi)
    N = np.empty((len(xi), 32)); dN = np.empty((len(xi), 32, 3))
    assert emu.lib.emu_shape_functions(_p(xi, _dp), len(xi), _p(N, _dp), _p(dN, _dp)) == 0
    assert ref_check("ref_grid_queries/box_split_N_dN", (N, dN), None, nan_equal=False)


def test_emulated_density_map_equals_reference_tool_output(emu, orc):
    """GenerateDensityMap --no-reduction of the reference (field 1 of the golden .cdm) from field 0 through the K3 kernel code, every
    node; and the predicate branch against the oracle"""
    g = read_cdf(os.path.join(GOLDEN, "ref_sphere_noreduction.cdm"))
    h, keep = emu.field(orc, g, 0)
    n = len(g["nodes"][0])
    out = np.full(n, np.nan)
    assert emu.lib.emu_density_map(h, 0.15, 1000.0, 1, 0, n, _p(out, _dp)) == 0
    assert bits_equal(out, g["nodes"][1])
    # predicate on, a node sub-range
    gd, res = keep[0], keep[1]
    l0, l1 = n // 5, n // 5 + 900
    want = orc.density_map(gd, res, g["nodes"][0], 0.15, 1000.0, False, l0, l1)
    part = np.full(l1 - l0, np.nan)
    assert emu.lib.emu_density_map(h, 0.15, 1000.0, 0, l0, l1, _p(part, _dp)) == 0
    assert bits_equal(part, want) and (part == DBL_MAX).any()
    emu.lib.emu_field_destroy(h)


def test_interpolate_fuzz_against_reference_class():
    """a short run of tools/k2_fuzz.py: random anisotropic grids and fields (DBL_MAX sentinels, reduced fields), queries on cell faces / domain
    corners / outside / non-finite -- emulated interpolate kernel == the reference class, value, gradient and value-only, bit for bit"""
    import subprocess
    import sys
    if not os.path.exists(LIBS[0]):
        pytest.skip("needs build/bin/libk23emu.so")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "k2_fuzz.py"), "24", "5"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_density_map_fuzz_against_oracle(emu):
    """a short run of tools/k3_fuzz.py on each emulated build (default, K3_FAST_DIV): random grids / fields / support radii / node ranges"""
    import subprocess
    import sys
    so = LIBS[0] if "knobs" not in emu.lib._name else LIBS[1]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "k3_fuzz.py"), "10", "3", so], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
