"""The product's K1 device code and launchers (discregrid_b200/csrc/k1_sdf.cu), compiled for the CPU by tests/emu (lanes of a warp as
fibers, warp votes resolved exactly) and compared with the oracle / the reference's golden vectors bit for bit -- the kernel logic is
therefore exercised by the CPU suite too (the real GPU runs are tests/test_gpu_k1_sdf.py).  What is emulated is the logic, not the
device's fp32 filter arithmetic, which by construction cannot change a result."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, bits_equal, grid_for
from test_oracle_golden import read_cdf, read_obj

# default knobs, the knob variants (K1_VOTE_REDUX + K1_BRICK_AUTO), the wavefront kernel, the per-lane kernel and the packet walk (K1_PACKET); DG_K1_EMU_LIB adds any other build of tests/emu/k1_emu.cpp
LIBS = [os.path.join(ROOT, "build", "bin", n) for n in ("libk1emu.so", "libk1emu_knobs.so", "libk1emu_wave.so", "libk1emu_perlane.so", "libk1emu_packet.so")] + \
       ([os.environ["DG_K1_EMU_LIB"]] if os.environ.get("DG_K1_EMU_LIB") else [])
_dp, _u32p, _i32p, _u64p = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int32), C.POINTER(C.c_uint64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


class Emu:
    def __init__(self, so):
        if not os.path.exists(so):
            pytest.skip(f"{so} not built (make cpp)")
        self.lib = C.CDLL(so)
        self.lib.emu_mesh_create.restype = C.c_void_p
        self.lib.emu_mesh_create.argtypes = [_dp, C.c_uint64, _u32p, C.c_uint64]
        self.lib.emu_mesh_destroy.argtypes = [C.c_void_p]
        self.lib.emu_sample_sdf.argtypes = [C.c_void_p, _dp, _u32p, C.c_double, C.c_uint64, C.c_uint64, _dp]
        self.lib.emu_sample_interleaved.argtypes = [C.c_void_p, _dp, _u32p, C.c_double, C.c_uint32, C.c_uint32, _dp, _u64p]
        self.lib.emu_unpack_interleaved.argtypes = [_dp, _u32p, C.c_uint32, _dp, _dp]
        self.lib.emu_sample_slab.argtypes = [C.c_void_p, _dp, _u32p, C.c_double, _u32p, _u32p, _dp]
        self.lib.emu_mesh_distance.argtypes = [C.c_void_p, _dp, C.c_uint64, C.c_int, _dp, _dp, _i32p, _i32p]
        self.lib.emu_node_positions.argtypes = [_dp, _u32p, C.c_uint64, C.c_uint64, _dp]
        self.lib.emu_build_cells.argtypes = [_dp, _u32p, C.c_uint64, C.c_uint64, _u32p]

    def mesh(self, V, F):
        V = np.ascontiguousarray(V, np.float64); F = np.ascontiguousarray(F, np.uint32)
        h = self.lib.emu_mesh_create(_p(V, _dp), len(V), _p(F, _u32p), len(F))
        assert h
        return h

    def sample(self, h, gd, res, l0, l1, sign=1.0):
        out = np.full(l1 - l0, np.nan)
        assert self.lib.emu_sample_sdf(h, _p(gd, _dp), _p(res, _u32p), sign, l0, l1, _p(out, _dp)) == 0
        return out


@pytest.fixture(scope="module", params=LIBS, ids=[os.path.basename(p) for p in LIBS])
def emu(request):
    return Emu(request.param)


def test_emulated_kernel_reproduces_box_cdf(emu, orc):
    """the reference's only golden vector, through the product's kernel code on the CPU: all 1296 coefficients and the connectivity"""
    g = read_cdf(os.path.join(GOLDEN, "box.cdf"))
    V, F = read_obj(os.path.join(GOLDEN, "box.obj"))
    gd, res = orc.grid_desc(g["mn"], g["mx"], g["res"], g["cell"], g["inv"])
    h = emu.mesh(V, F)
    assert bits_equal(emu.sample(h, gd, res, 0, len(g["nodes"][0])), g["nodes"][0])
    cells = np.zeros((125, 32), np.uint32)
    assert emu.lib.emu_build_cells(_p(gd, _dp), _p(res, _u32p), 0, 125, _p(cells, _u32p)) == 0
    assert np.array_equal(cells, g["cells"][0])
    emu.lib.emu_mesh_destroy(h)


@pytest.mark.parametrize("res", [(9, 8, 7), (16, 5, 3)])
def test_emulated_node_loop_ranges_and_shardings(emu, orc, res):
    """whole grid, ragged node ranges (masked bricks), the slab form and the interleaved deal + unpack: all equal to the oracle"""
    import discregrid_b200 as dg
    t = dg.bumpy_torus(24, 20, 1.0, 0.4, 0.05, 7, 5)
    mn, mx, gd, r = grid_for(orc, t.vertices, res)
    want = orc.mesh(t.vertices, t.faces).sample_sdf(gd, r)
    n = len(want)
    h = emu.mesh(t.vertices, t.faces)
    assert bits_equal(emu.sample(h, gd, r, 0, n), want)
    for (a, b) in [(0, 1), (5, 77), (n // 3, n // 3 + 1000), (n - 13, n)]:
        b = min(b, n)
        assert bits_equal(emu.sample(h, gd, r, a, b, sign=-1.0), -want[a:b])
    # interleaved deal over 3 parts + unpack
    se = C.c_uint64()
    assert emu.lib.emu_sample_interleaved(h, _p(gd, _dp), _p(r, _u32p), 1.0, 0, 3, None, C.byref(se)) == 0
    slots = np.full(3 * se.value, np.nan)
    for part in range(3):
        assert emu.lib.emu_sample_interleaved(h, _p(gd, _dp), _p(r, _u32p), 1.0, part, 3, _p(slots, _dp), C.byref(se)) == 0
    full = np.full(n, np.nan)
    assert emu.lib.emu_unpack_interleaved(_p(gd, _dp), _p(r, _u32p), 3, _p(slots, _dp), _p(full, _dp)) == 0
    assert bits_equal(full, want)
    # slab form: whole slow-plane pairs of each of the four node arrays, three parts, written at their final positions
    nx, ny, nz = res
    ds = [nz + 1, nz + 1, nx + 1, ny + 1]                         # slow dimension of the vertex / x-edge / y-edge / z-edge arrays
    full2 = np.full(n, np.nan)
    for part in range(3):
        pb = np.array([2 * ((((d + 1) // 2) * part) // 3) for d in ds], np.uint32)
        pe = np.array([min(d, 2 * ((((d + 1) // 2) * (part + 1)) // 3)) for d in ds], np.uint32)
        assert emu.lib.emu_sample_slab(h, _p(gd, _dp), _p(r, _u32p), 1.0, _p(pb, _u32p), _p(pe, _u32p), _p(full2, _dp)) == 0
    assert bits_equal(full2, want)
    # node positions
    x = np.zeros((n, 3))
    assert emu.lib.emu_node_positions(_p(gd, _dp), _p(r, _u32p), 0, n, _p(x, _dp)) == 0
    assert bits_equal(x, orc.node_positions(gd, r, 0, n))
    emu.lib.emu_mesh_destroy(h)


def test_emulated_distance_queries_match_reference_header(emu):
    """mesh_distance_kernel on the CPU vs results of the reference's own TriangleMeshDistance.h (golden): distance, nearest point,
    entity and triangle, signed and unsigned, including points on the surface"""
    import discregrid_b200 as dg
    q = np.load(os.path.join(GOLDEN, "ref_torus_queries.npz"))
    t = dg.bumpy_torus(*[int(a) if i < 2 or i > 4 else float(a) for i, a in enumerate(q["torus_args"])])
    h = emu.mesh(t.vertices, t.faces)
    x = np.ascontiguousarray(q["x"][:1500]); n = len(x)
    dist = np.zeros(n); near = np.zeros((n, 3)); ent = np.zeros(n, np.int32); tri = np.zeros(n, np.int32)
    assert emu.lib.emu_mesh_distance(h, _p(x, _dp), n, 1, _p(dist, _dp), _p(near, _dp), _p(ent, _i32p), _p(tri, _i32p)) == 0
    assert bits_equal(dist, q["distance"][:n]) and bits_equal(near, q["nearest"][:n])
    assert np.array_equal(ent, q["entity"][:n]) and np.array_equal(tri, q["triangle"][:n])
    assert emu.lib.emu_mesh_distance(h, _p(x, _dp), n, 0, _p(dist, _dp), None, None, None) == 0
    assert bits_equal(dist, q["unsigned"][:n])
    emu.lib.emu_mesh_destroy(h)
    s = np.load(os.path.join(GOLDEN, "ref_sphere_surface.npz"))
    a = s["sphere_args"]
    sp = dg.uv_sphere(int(a[0]), int(a[1]), float(a[2]), (float(a[3]), float(a[4]), float(a[5])))
    h = emu.mesh(sp.vertices, sp.faces)
    xs = np.ascontiguousarray(s["x"]); n = len(xs)
    dist = np.zeros(n); near = np.zeros((n, 3)); ent = np.zeros(n, np.int32); tri = np.zeros(n, np.int32)
    assert emu.lib.emu_mesh_distance(h, _p(xs, _dp), n, 1, _p(dist, _dp), _p(near, _dp), _p(ent, _i32p), _p(tri, _i32p)) == 0
    assert bits_equal(dist, s["distance"]) and bits_equal(near, s["nearest"]) and np.array_equal(ent, s["entity"]) and np.array_equal(tri, s["triangle"])
    emu.lib.emu_mesh_destroy(h)


def _rand_mesh(rng, n_tri, scale=1.0, offset=0.0, degenerate=False):
    V = rng.standard_normal((n_tri + 2, 3)) * scale + offset
    F = np.array([[i, i + 1, i + 2] for i in range(n_tri)], np.uint32)        # a strip: neighbours share edges and vertices (ties)
    if degenerate and n_tri >= 3:
        V[3] = V[2]                                                            # zero-length edge -> zero-area triangles
        F[-1] = [0, 0, 1]                                                      # a triangle with a repeated vertex
    return np.ascontiguousarray(V), F


@pytest.mark.parametrize("n_tri,scale,offset,degenerate", [(1, 1.0, 0.0, False), (2, 1.0, 0.0, False), (3, 1.0, 0.0, False), (7, 1e-9, 0.0, False),
                                                           (40, 1.0, 1e9, False), (33, 1e6, -3e7, False), (9, 1.0, 0.0, True), (64, 1.0, 0.0, True)])
def test_emulated_queries_on_awkward_meshes_vs_reference_header(emu, n_tri, scale, offset, degenerate):
    """corner cases against the reference's own TriangleMeshDistance.h (its results stored as digests, oracle_api.ref_check): one- and
    two-triangle meshes (the root is a leaf / has leaf children), tiny and huge coordinates (the fp32 filter's error bound scales with them),
    far-away and non-finite queries (filter switched off / NaN comparisons), degenerate triangles (0/0 in the reference's formulas): same
    distance bits -- NaN for NaN --, same nearest point, entity and triangle"""
    from oracle_api import RefMesh, ref_check
    rng = np.random.default_rng(1000 + n_tri)
    V, F = _rand_mesh(rng, n_tri, scale, offset, degenerate)
    x = np.concatenate([rng.standard_normal((300, 3)) * scale * 2 + offset,                    # around the mesh
                        V[:min(len(V), 20)],                                                  # exactly on vertices
                        0.5 * (V[F[:, 0]] + V[F[:, 1]])[:20],                                  # on edges
                        rng.standard_normal((40, 3)) * scale * 1e6 + offset,                   # far
                        np.array([[1e19, -1e19, 3e18], [0.0, 0.0, 0.0], [-0.0, 0.0, -0.0]])])
    x = np.ascontiguousarray(x)
    # queries for which the reference accepts no triangle (NaN, infinite, or so large that the squared distance overflows) make it index
    # triangles[-1] (undefined behaviour: it crashes for some meshes): not sent to the reference; the kernel must answer DBL_MAX / -1
    lost = np.ascontiguousarray(np.array([[1e300, 0, 0], [np.nan, 0, 0], [np.inf, 1, 2], [0, -np.inf, 0]]))
    h = emu.mesh(V, F)
    for signed in (1, 0):
        n = len(x)
        dist = np.zeros(n); near = np.zeros((n, 3)); ent = np.zeros(n, np.int32); tri = np.zeros(n, np.int32)
        assert emu.lib.emu_mesh_distance(h, _p(x, _dp), n, signed, _p(dist, _dp), _p(near, _dp), _p(ent, _i32p), _p(tri, _i32p)) == 0
        assert (tri >= 0).all()                                                # the reference finds a triangle for every one of these
        key = f"k1_awkward_mesh/{n_tri}/{scale!r}/{offset!r}/{degenerate}/signed={signed}"
        assert ref_check(key, (dist, near, ent, tri), lambda: RefMesh(V, F).distance(x, signed=bool(signed))), key
        d2 = np.zeros(len(lost)); t2 = np.zeros(len(lost), np.int32)
        assert emu.lib.emu_mesh_distance(h, _p(lost, _dp), len(lost), signed, _p(d2, _dp), None, None, _p(t2, _i32p)) == 0
        assert (d2 == np.finfo(np.float64).max).all() and (t2 == -1).all()
    emu.lib.emu_mesh_destroy(h)


def test_tie_rich_fuzz_against_reference_header():
    """a short run of tools/k1_fuzz.py (regular coplanar grids, cubes / octahedra with lattice-aligned queries, duplicated triangles,
    slivers, random soups at random scales): emulated kernel == reference header in distance bits, nearest point, entity, triangle id"""
    import subprocess
    import sys
    so = LIBS[0]
    if not os.path.exists(so):
        pytest.skip("needs build/bin/libk1emu.so")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "k1_fuzz.py"), "42", "7", so], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


@pytest.mark.parametrize("name", ["libk1emu.so", "libk1emu_packet.so"])
def test_tie_rich_grid_fuzz_node_loop_against_reference_header(name):
    """tools/k1_fuzz.py in grid mode: the addFunction node loop (bricks of lattice nodes; for libk1emu_packet.so the packet walk with its
    tie replay, certificates and per-lane fallback) on half-integer lattices through coplanar grids, cubes, octahedra, duplicated triangles,
    slivers and random soups == sign * the reference header's signed distance at the node positions, bit for bit"""
    import subprocess
    import sys
    so = os.path.join(ROOT, "build", "bin", name)
    if not os.path.exists(so):
        pytest.skip("needs build/bin/" + name)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "k1_fuzz.py"), "21", "11", so, "grid"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "0 mismatches" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_node_loop_on_a_mesh_with_non_finite_vertices(emu, orc):
    """NaN / inf vertices: the reference's sphere tests then compare false and whole subtrees go unvisited -- nothing an order-free search may
    assume.  The host builder marks such a mesh (half_extent = +inf), every fp32 filter switches off and the packet walk hands all its lanes to
    the per-lane walk: node loop == reference header bit for bit"""
    from oracle_api import RefMesh, ref_check
    V = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1], [np.nan, 2, 2], [3, 3, np.inf], [2, 2, 2]], float)
    F = np.array([[0, 2, 4], [2, 1, 4], [1, 3, 4], [3, 0, 4], [2, 0, 5], [1, 2, 5], [3, 1, 5], [0, 3, 5], [6, 0, 2], [7, 8, 4]], np.uint32)
    gd, r = orc.grid_desc(np.array([-2.0, -2, -2]), np.array([2.0, 2, 2]), (8, 8, 8))
    nn = orc.num_nodes(r)
    xs = np.empty((nn, 3))
    emu.lib.emu_node_positions(_p(gd, _dp), _p(r, _u32p), 0, nn, _p(xs, _dp))
    h = emu.mesh(V, F)
    got = emu.sample(h, gd, r, 0, nn)
    assert ref_check("k1_non_finite_vertices/8x8x8", (got,), lambda: (RefMesh(V, F).distance(xs, signed=True)[0],), nan_equal=False)
    emu.lib.emu_mesh_destroy(h)


def test_emulated_launch_order(emu, orc):
    """the per-lane sampling kernel takes its blocks in launch order, every block exactly once (the wavefront kernel hands out bricks
    through a counter instead and has no block order)"""
    import discregrid_b200 as dg
    if "wave" in emu.lib._name:
        pytest.skip("the wavefront kernel hands out bricks through a counter: there is no block order")
    emu.lib.emu_block_trace.restype = C.c_uint64
    emu.lib.emu_block_trace.argtypes = [_u32p, C.c_uint64]
    t = dg.bumpy_torus(24, 20, 1.0, 0.4, 0.05, 7, 5)
    mn, mx, gd, r = grid_for(orc, t.vertices, (20, 20, 20))
    nv = 21 ** 3
    h = emu.mesh(t.vertices, t.faces)
    buf = np.zeros(1 << 16, np.uint32)
    emu.lib.emu_block_trace(_p(buf, _u32p), len(buf))                      # clear
    emu.sample(h, gd, r, 0, nv)
    n = emu.lib.emu_block_trace(_p(buf, _u32p), len(buf))
    order = buf[:n].astype(np.int64)
    assert n > 100 and np.array_equal(order, np.arange(n))
    emu.lib.emu_mesh_destroy(h)
