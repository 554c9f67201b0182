"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when built, the reference's own
TriangleMeshDistance.h (oracle/_ref/libdgref.so).  TEST INFRASTRUCTURE ONLY -- the product package
(discregrid_b200/) never imports this module."""
import ctypes as C
import hashlib
import json
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "liboracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libdgref.so")
REF_RESOURCES = os.path.join(ROOT, "oracle", "_ref", "resources")
REF_GRID_SO = os.path.join(ROOT, "oracle", "_ref", "libdiscregrid_ref.so")
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bin")
REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.json")

_dp = C.POINTER(C.c_double)
_u32p = C.POINTER(C.c_uint32)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def digest(arrays, nan_equal=True):
    """sha256 over a tuple of arrays (length and values; integers as int64, floats as float64).  nan_equal: every NaN is replaced by
    the same NaN first, so that two results have the same digest exactly when they are equal bit for bit, any NaN matching any NaN."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.asarray(a).ravel()
        if a.dtype.kind == "f":
            a = a.astype(np.float64)
            if nan_equal:
                a = np.where(np.isnan(a), np.nan, a)
        else:
            a = a.astype(np.int64)
        h.update(b"%d:" % len(a))
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


_digests = None


def ref_check(key, got, live, nan_equal=True):
    """True when `got` (a tuple of arrays) equals the reference's result on the same inputs.  The reference's results on the test inputs are
    kept as digests in tests/golden/ref_digests.json, so that the comparison needs no build of the reference.  `live` computes the result
    with the reference itself (oracle/_ref); it runs instead when `key` is not stored, and DG_RECORD_REF_DIGESTS=1 makes it run and store its
    digest under `key` (tests/golden/make_golden.py).  live=None: the stored digest only (written by make_golden.py itself)."""
    global _digests
    if _digests is None:
        _digests = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
    record = os.environ.get("DG_RECORD_REF_DIGESTS") == "1"
    if key in _digests and (not record or live is None):
        return digest(got, nan_equal) == _digests[key]
    if live is None:
        raise KeyError(f"no stored digest of the reference's result for {key!r}")
    try:
        want = digest(live(), nan_equal)
    except OSError as ex:
        raise KeyError(f"no stored digest of the reference's result for {key!r}, and the reference is not built (oracle/_ref)") from ex
    if record:
        _digests = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
        _digests[key] = want
        with open(REF_DIGESTS, "w") as f:
            json.dump(_digests, f, indent=0, sort_keys=True)
            f.write("\n")
    return digest(got, nan_equal) == want


class _MeshBase:
    """Common wrapper over the {orc,ref}_mesh_* entry points."""

    def __init__(self, lib, prefix, V, F):
        self._lib, self._px = lib, prefix
        self.V, self.F = _f64(V).reshape(-1, 3), _u32(F).reshape(-1, 3)
        f = getattr(lib, prefix + "mesh_create")
        f.restype = C.c_void_p
        f.argtypes = [_dp, C.c_uint64, _u32p, C.c_uint64]
        self.h = f(_p(self.V, _dp), len(self.V), _p(self.F, _u32p), len(self.F))
        if not self.h:
            raise ValueError("empty triangle list")

    def close(self):
        if getattr(self, "h", None):
            f = getattr(self._lib, self._px + "mesh_destroy")
            f.argtypes = [C.c_void_p]
            f(self.h)
            self.h = None

    __del__ = close

    def tree(self):
        f = getattr(self._lib, self._px + "mesh_num_nodes")
        f.restype = C.c_uint64
        f.argtypes = [C.c_void_p]
        n = f(self.h)
        sph = np.empty((n, 8), np.float64)
        kids = np.empty((n, 2), np.int32)
        g = getattr(self._lib, self._px + "mesh_tree")
        g.argtypes = [C.c_void_p, _dp, _i32p]
        g(self.h, _p(sph, _dp), _p(kids, _i32p))
        return sph, kids

    def pseudonormals(self):
        tri = np.empty((len(self.F), 3)); edge = np.empty((len(self.F), 3, 3)); vert = np.empty((len(self.V), 3))
        g = getattr(self._lib, self._px + "mesh_pseudonormals")
        g.argtypes = [C.c_void_p, _dp, _dp, _dp]
        g(self.h, _p(tri, _dp), _p(edge, _dp), _p(vert, _dp))
        return tri, edge, vert

    def distance(self, x, signed=True):
        x = _f64(x).reshape(-1, 3)
        n = len(x)
        dist = np.empty(n); near = np.empty((n, 3)); ent = np.empty(n, np.int32); tri = np.empty(n, np.int32)
        g = getattr(self._lib, self._px + "mesh_distance")
        g.argtypes = [C.c_void_p, _dp, C.c_uint64, C.c_int, _dp, _dp, _i32p, _i32p]
        g(self.h, _p(x, _dp), n, int(signed), _p(dist, _dp), _p(near, _dp), _p(ent, _i32p), _p(tri, _i32p))
        return dist, near, ent, tri


class Oracle:
    """The restated oracle (oracle/dg_oracle.cpp)."""

    def __init__(self):
        if not os.path.exists(ORACLE_SO):
            raise RuntimeError("oracle/liboracle.so missing: run `make -C oracle oracle` (or __graft_entry__.build())")
        self.lib = C.CDLL(ORACLE_SO)
        self.lib.orc_num_nodes.restype = C.c_uint64
        self.lib.orc_max_threads.restype = C.c_int

    def mesh(self, V, F):
        return OracleMesh(self, V, F)

    def max_threads(self):
        return self.lib.orc_max_threads()

    @staticmethod
    def grid_desc(mn, mx, res, cell=None, inv=None):
        """12 doubles (min, max, cell, inv) + res[3]."""
        mn, mx = _f64(mn), _f64(mx)
        res = _u32(res)
        if cell is None:
            cell = np.empty(3); inv = np.empty(3)
            lib = C.CDLL(ORACLE_SO)
            lib.orc_grid_constants(_p(mn, _dp), _p(mx, _dp), _p(res, _u32p), _p(cell, _dp), _p(inv, _dp))
        return np.concatenate([mn, mx, _f64(cell), _f64(inv)]), res

    def generate_sdf_domain(self, V):
        V = _f64(V).reshape(-1, 3)
        mn = np.empty(3); mx = np.empty(3)
        self.lib.orc_generate_sdf_domain(_p(V, _dp), C.c_uint64(len(V)), _p(mn, _dp), _p(mx, _dp))
        return mn, mx

    def num_nodes(self, res):
        res = _u32(res)
        return int(self.lib.orc_num_nodes(_p(res, _u32p)))

    def node_positions(self, gd, res, l0, l1):
        x = np.empty((l1 - l0, 3))
        self.lib.orc_node_positions(_p(gd, _dp), _p(res, _u32p), C.c_uint64(l0), C.c_uint64(l1), _p(x, _dp))
        return x

    def node_positions_at(self, gd, res, ids):
        ids = np.ascontiguousarray(ids, dtype=np.uint64)
        x = np.empty((len(ids), 3))
        self.lib.orc_node_positions_at(_p(gd, _dp), _p(res, _u32p), ids.ctypes.data_as(C.POINTER(C.c_uint64)), C.c_uint64(len(ids)), _p(x, _dp))
        return x

    def build_cells(self, res, c0=0, c1=None):
        res = _u32(res)
        if c1 is None:
            c1 = int(res[0]) * int(res[1]) * int(res[2])
        cells = np.empty((c1 - c0, 32), np.uint32)
        self.lib.orc_build_cells(_p(res, _u32p), C.c_uint64(c0), C.c_uint64(c1), _p(cells, _u32p))
        return cells

    def shape_functions(self, xi, grad=True):
        xi = _f64(xi).reshape(-1, 3)
        N = np.empty((len(xi), 32)); dN = np.empty((len(xi), 32, 3)) if grad else None
        self.lib.orc_shape_functions(_p(xi, _dp), C.c_uint64(len(xi)), _p(N, _dp), _p(dN, _dp))
        return N, dN

    def interpolate(self, gd, res, nodes, x, grad=True, cells=None, cell_map=None, nthreads=0):
        x = _f64(x).reshape(-1, 3)
        nodes = _f64(nodes)
        cells = None if cells is None else _u32(cells)
        cell_map = None if cell_map is None else _u32(cell_map)
        # the reference returns before touching *gradient for out-of-domain / removed cells (:981-982, :993-994): the
        # caller's value survives.  The batch API defines that value as 0, so the oracle's buffer starts zeroed.
        phi = np.empty(len(x)); g = np.zeros((len(x), 3)) if grad else None
        self.lib.orc_interpolate(_p(gd, _dp), _p(res, _u32p), _p(nodes, _dp), _p(cells, _u32p), _p(cell_map, _u32p),
                                 _p(x, _dp), C.c_uint64(len(x)), _p(phi, _dp), _p(g, _dp), C.c_int(nthreads))
        return phi, g

    def density_map(self, gd, res, nodes, h, rho0, no_reduction, l0, l1, cells=None, cell_map=None, nthreads=0):
        nodes = _f64(nodes)
        cells = None if cells is None else _u32(cells)
        cell_map = None if cell_map is None else _u32(cell_map)
        out = np.empty(l1 - l0)
        self.lib.orc_density_map(_p(gd, _dp), _p(res, _u32p), _p(nodes, _dp), _p(cells, _u32p), _p(cell_map, _u32p),
                                 C.c_double(h), C.c_double(rho0), C.c_int(int(no_reduction)), C.c_uint64(l0),
                                 C.c_uint64(l1), _p(out, _dp), C.c_int(nthreads))
        return out


class OracleMesh(_MeshBase):
    def __init__(self, orc, V, F):
        self.orc = orc
        super().__init__(orc.lib, "orc_", V, F)

    def flags(self):
        self._lib.orc_mesh_flags.argtypes = [C.c_void_p]
        return self._lib.orc_mesh_flags(self.h)

    def sample_sdf(self, gd, res, sign=1.0, l0=0, l1=None, nthreads=0):
        if l1 is None:
            l1 = self.orc.num_nodes(res)
        out = np.empty(l1 - l0)
        f = self._lib.orc_sample_sdf
        f.argtypes = [C.c_void_p, _dp, _u32p, C.c_double, C.c_uint64, C.c_uint64, _dp, C.c_int]
        f(self.h, _p(gd, _dp), _p(res, _u32p), sign, l0, l1, _p(out, _dp), nthreads)
        return out

    def stats(self, x):
        x = _f64(x).reshape(-1, 3)
        v = C.c_int64(); l = C.c_int64()
        f = self._lib.orc_mesh_stats
        f.argtypes = [C.c_void_p, _dp, C.c_uint64, _i64p, _i64p]
        f(self.h, _p(x, _dp), len(x), C.byref(v), C.byref(l))
        return v.value / len(x), l.value / len(x)


def have_ref():
    return os.path.exists(REF_SO)


class RefMesh(_MeshBase):
    """The reference's own TriangleMeshDistance (oracle/_ref/libdgref.so)."""

    def __init__(self, V, F):
        super().__init__(C.CDLL(REF_SO), "ref_", V, F)

    def sample_points(self, x, sign=1.0, nthreads=0):
        x = _f64(x).reshape(-1, 3)
        out = np.empty(len(x))
        f = self._lib.ref_sample_points
        f.argtypes = [C.c_void_p, _dp, C.c_uint64, C.c_double, _dp, C.c_int]
        f(self.h, _p(x, _dp), len(x), sign, _p(out, _dp), nthreads)
        return out


def have_ref_grid():
    return os.path.exists(REF_GRID_SO)


class RefGrid:
    """The reference's own CubicLagrangeDiscreteGrid (unmodified sources compiled against the Eigen stand-in, oracle/Makefile)."""

    def __init__(self, path):
        self.lib = C.CDLL(REF_GRID_SO)
        self.lib.refg_load.restype = C.c_void_p
        self.lib.refg_load.argtypes = [C.c_char_p]
        self.h = self.lib.refg_load(path.encode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.refg_destroy.argtypes = [C.c_void_p]
            self.lib.refg_destroy(self.h)
            self.h = None

    __del__ = close

    def interpolate(self, field, x, grad=True, nthreads=0):
        x = _f64(x).reshape(-1, 3)
        phi = np.empty(len(x)); g = np.zeros((len(x), 3)) if grad else None
        f = self.lib.refg_interpolate
        f.argtypes = [C.c_void_p, C.c_uint, _dp, C.c_uint64, _dp, _dp, C.c_int]
        f(self.h, field, _p(x, _dp), len(x), _p(phi, _dp), _p(g, _dp), nthreads)
        return phi, g

    def reduce_window(self, field, lo, hi):
        """reduceField(field, lo <= v <= hi); returns the seconds the reference's call took"""
        f = self.lib.refg_reduce_window
        f.argtypes = [C.c_void_p, C.c_uint, C.c_double, C.c_double]; f.restype = C.c_double
        return f(self.h, field, lo, hi)

    def save(self, path):
        self.lib.refg_save.argtypes = [C.c_void_p, C.c_char_p]
        self.lib.refg_save(self.h, path.encode())

    def split(self, field, x):
        x = _f64(x).reshape(-1, 3); n = len(x)
        ok = np.zeros(n, np.int32); N = np.zeros((n, 32)); dN = np.zeros((n, 32, 3)); c0 = np.zeros((n, 3))
        cell = np.zeros((n, 32), np.uint32); phi = np.zeros(n); grad = np.zeros((n, 3))
        f = self.lib.refg_split
        f.argtypes = [C.c_void_p, C.c_uint, _dp, C.c_uint64, _i32p, _dp, _dp, _dp, _u32p, _dp, _dp]
        f(self.h, field, _p(x, _dp), n, _p(ok, _i32p), _p(N, _dp), _p(dN, _dp), _p(c0, _dp), _p(cell, _u32p), _p(phi, _dp), _p(grad, _dp))
        return ok, N, dN, c0, cell, phi, grad


class RefAddFunction:
    """The reference's REAL CubicLagrangeDiscreteGrid::addFunction with the GenerateSDF functor (oracle/ref_grid_wrapper.cpp:
    refg_md_create / refg_add_function_sdf; cmd/generate_sdf/main.cpp:74,92-105, cubic_lagrange_discrete_grid.cpp:780-899)."""

    def __init__(self, V, F):
        self.lib = C.CDLL(REF_GRID_SO)
        V, F = _f64(V).reshape(-1, 3), _u32(F).reshape(-1, 3)
        self.lib.refg_md_create.restype = C.c_void_p
        self.lib.refg_md_create.argtypes = [_dp, C.c_uint64, _u32p, C.c_uint64]
        self.h = self.lib.refg_md_create(_p(V, _dp), len(V), _p(F, _u32p), len(F))
        self.lib.refg_add_function_sdf.restype = C.c_double
        self.lib.refg_add_function_sdf.argtypes = [C.c_void_p, _dp, _dp, _u32p, C.c_int, C.c_int, _dp, _u32p, C.POINTER(C.c_uint64)]
        self.lib.refg_omp_max_threads.restype = C.c_int

    def max_threads(self):
        return self.lib.refg_omp_max_threads()

    def add_function(self, mn, mx, res, invert=False, nthreads=0, want_nodes=False, want_cells=False):
        """-> (seconds of the reference's addFunction call, nodes or None, cells or None)"""
        mn, mx, res = _f64(mn), _f64(mx), _u32(res)
        nx, ny, nz = (int(r) for r in res)
        n_nodes = (nx + 1) * (ny + 1) * (nz + 1) + 2 * (nx * (ny + 1) * (nz + 1) + (nx + 1) * ny * (nz + 1) + (nx + 1) * (ny + 1) * nz)
        nodes = np.empty(n_nodes) if want_nodes else None
        cells = np.empty((nx * ny * nz, 32), np.uint32) if want_cells else None
        n_out = C.c_uint64()
        dt = self.lib.refg_add_function_sdf(self.h, _p(mn, _dp), _p(mx, _dp), _p(res, _u32p), int(invert), int(nthreads),
                                            _p(nodes, _dp), _p(cells, _u32p), C.byref(n_out))
        assert n_out.value == n_nodes
        return dt, nodes, cells

    def close(self):
        if getattr(self, "h", None):
            self.lib.refg_md_destroy.argtypes = [C.c_void_p]
            self.lib.refg_md_destroy(self.h)
            self.h = None

    __del__ = close


class RefGridInMemory(RefGrid):
    """RefGrid over a coefficient array handed over in memory (oracle/ref_grid_wrapper.cpp: refg_grid_from_nodes)."""

    def __init__(self, mn, mx, res, nodes, nthreads=0):
        self.lib = C.CDLL(REF_GRID_SO)
        mn, mx, res, nodes = _f64(mn), _f64(mx), _u32(res), _f64(nodes)
        self.lib.refg_grid_from_nodes.restype = C.c_void_p
        self.lib.refg_grid_from_nodes.argtypes = [_dp, _dp, _u32p, _dp, C.c_uint64, C.c_int]
        self.h = self.lib.refg_grid_from_nodes(_p(mn, _dp), _p(mx, _dp), _p(res, _u32p), _p(nodes, _dp), len(nodes), int(nthreads))
        if not self.h:
            raise ValueError("node count does not match the grid")
