#!/usr/bin/env python
"""Parity fuzzer (CPU): the product's K1 kernel code run by tests/emu (build/bin/libk1emu*.so) against the reference's own
TriangleMeshDistance.h (oracle/_ref/libdgref.so) on meshes built to provoke exact ties and awkward arithmetic -- regular grids of coplanar
triangles, cubes / octahedra with queries on symmetry planes, duplicated triangles, slivers, lattice-aligned queries -- signed and unsigned,
distance bits, nearest point, entity and triangle id.  usage: tools/k1_fuzz.py [rounds=200] [seed=0] [lib=libk1emu.so] [points|grid]
mode `grid` runs the addFunction NODE LOOP (sdf_sample_nodes_kernel: bricks of lattice nodes, the packet walk when built with K1_PACKET) on
lattices laid over the same meshes -- half-integer lattices through the symmetric ones -- and compares sign * distance bit for bit with the
reference header evaluated at the node positions.  The reference's results come from tests/golden/ref_digests.json where they are stored
for a case (oracle_api.ref_check), from oracle/_ref otherwise; a mismatch is reported per case."""
import ctypes as C, os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle_api import RefMesh, ref_check
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 200
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
so = sys.argv[3] if len(sys.argv) > 3 else os.path.join(ROOT, "build", "bin", "libk1emu.so")
mode = sys.argv[4] if len(sys.argv) > 4 else "points"
lib = C.CDLL(so)
dp, u32p, i32p = C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int32)
lib.emu_mesh_create.restype = C.c_void_p
lib.emu_mesh_create.argtypes = [dp, C.c_uint64, u32p, C.c_uint64]
lib.emu_mesh_destroy.argtypes = [C.c_void_p]
lib.emu_mesh_distance.argtypes = [C.c_void_p, dp, C.c_uint64, C.c_int, dp, dp, i32p, i32p]
lib.emu_sample_sdf.argtypes = [C.c_void_p, dp, u32p, C.c_double, C.c_uint64, C.c_uint64, dp]
lib.emu_node_positions.argtypes = [dp, u32p, C.c_uint64, C.c_uint64, dp]
rng = np.random.default_rng(seed)


def grid_mesh(nx, ny, jitter=0.0, z=0.0):
    xs, ys = np.meshgrid(np.arange(nx + 1, dtype=float), np.arange(ny + 1, dtype=float), indexing="ij")
    V = np.stack([xs.ravel(), ys.ravel(), np.full(xs.size, z)], 1)
    V[:, :2] += jitter * rng.standard_normal((len(V), 2))
    F = []
    for i in range(nx):
        for j in range(ny):
            a, b, c, d = i * (ny + 1) + j, (i + 1) * (ny + 1) + j, (i + 1) * (ny + 1) + j + 1, i * (ny + 1) + j + 1
            F += [[a, b, c], [a, c, d]] if (i + j) % 2 else [[a, b, d], [b, c, d]]
    return V, np.array(F, np.uint32)


def cube(n=1):
    V = np.array([[x, y, z] for x in (0, 1) for y in (0, 1) for z in (0, 1)], float)
    F = np.array([[0, 1, 3], [0, 3, 2], [4, 6, 7], [4, 7, 5], [0, 4, 5], [0, 5, 1], [2, 3, 7], [2, 7, 6], [0, 2, 6], [0, 6, 4], [1, 5, 7], [1, 7, 3]], np.uint32)
    return V, F


def octa():
    V = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], float)
    F = np.array([[0, 2, 4], [2, 1, 4], [1, 3, 4], [3, 0, 4], [2, 0, 5], [1, 2, 5], [3, 1, 5], [0, 3, 5]], np.uint32)
    return V, F


def make_case(k):
    kind = k % 7
    if kind == 0: V, F = grid_mesh(int(rng.integers(1, 7)), int(rng.integers(1, 7)))
    elif kind == 1: V, F = grid_mesh(int(rng.integers(2, 6)), int(rng.integers(2, 6)), jitter=1e-3)
    elif kind == 2: V, F = cube()
    elif kind == 3: V, F = octa()
    elif kind == 4:                                              # two stacked sheets + duplicated triangles
        V1, F1 = grid_mesh(3, 3); V2, F2 = grid_mesh(3, 3, z=1.0)
        V = np.concatenate([V1, V2]); F = np.concatenate([F1, F2 + len(V1), F1[:4]])
    elif kind == 5:                                              # slivers and near-degenerate triangles
        n = int(rng.integers(3, 30)); V = rng.standard_normal((n + 2, 3)); V[:, 2] *= 1e-7
        F = np.array([[i, i + 1, i + 2] for i in range(n)], np.uint32)
    else:                                                        # random soup, random scale / offset
        n = int(rng.integers(1, 60)); sc = 10.0 ** rng.integers(-6, 7); off = rng.standard_normal(3) * sc * 10 ** rng.integers(0, 4)
        V = rng.standard_normal((3 * n, 3)) * sc + off; F = np.arange(3 * n, dtype=np.uint32).reshape(n, 3)
    V = np.ascontiguousarray(V, np.float64); F = np.ascontiguousarray(F, np.uint32)
    lo, hi = V.min(0), V.max(0); ext = np.maximum(hi - lo, 1e-12)
    q = [lo - 0.5 * ext + rng.random((150, 3)) * 2 * ext]
    lat = np.stack(np.meshgrid(*[np.linspace(lo[d] - ext[d], hi[d] + ext[d], 7) for d in range(3)], indexing="ij"), -1).reshape(-1, 3)
    q += [lat, V, 0.5 * (V[F[:, 0]] + V[F[:, 1]]), (V[F[:, 0]] + V[F[:, 1]] + V[F[:, 2]]) / 3.0]
    if kind in (0, 2, 3, 4):                                     # half-integer lattice: symmetric, tie-rich queries
        q.append(np.stack(np.meshgrid(*[np.arange(-1.0, 2.51, 0.5)] * 3, indexing="ij"), -1).reshape(-1, 3))
    return V, F, np.ascontiguousarray(np.concatenate(q))


bad = 0
total = 0
for k in range(rounds):
    V, F, x = make_case(k)
    h = lib.emu_mesh_create(V.ctypes.data_as(dp), len(V), F.ctypes.data_as(u32p), len(F))
    if mode == "grid":
        from oracle_api import Oracle
        lo, hi = V.min(0), V.max(0); ext = np.maximum(hi - lo, 1e-9)
        if k % 7 in (0, 2, 3, 4):                                 # nodes on the half-integer lattice: ties by symmetry
            mn = np.floor(lo) - 1.0; mx = mn + 4.0 * np.ceil((hi - mn + 1.0) / 4.0); res = tuple(int(r) for r in ((mx - mn) * 2))
        else:
            mn = lo - 0.3 * ext; mx = hi + 0.3 * ext; res = (9, 7, 6)
        gd, r = Oracle().grid_desc(mn, mx, res)
        nn = (res[0] + 1) * (res[1] + 1) * (res[2] + 1) + 2 * (res[0] * (res[1] + 1) * (res[2] + 1) + (res[0] + 1) * res[1] * (res[2] + 1) + (res[0] + 1) * (res[1] + 1) * res[2])
        xs = np.empty((nn, 3)); lib.emu_node_positions(gd.ctypes.data_as(dp), r.ctypes.data_as(u32p), 0, nn, xs.ctypes.data_as(dp))
        sign = 1.0 if k % 2 else -1.0
        got = np.full(nn, np.nan)
        assert lib.emu_sample_sdf(h, gd.ctypes.data_as(dp), r.ctypes.data_as(u32p), sign, 0, nn, got.ctypes.data_as(dp)) == 0
        total += nn
        key = f"k1_fuzz/grid/{seed}/{k}"
        if not ref_check(key, (got,), lambda: (sign * RefMesh(V, F).distance(xs, signed=True)[0],)):
            bad += 1
            print(f"MISMATCH {key} (kind {k % 7}, {len(F)} tris) grid {res}")
        lib.emu_mesh_destroy(h)
        continue
    n = len(x)
    for signed in (1, 0):
        d = np.zeros(n); nr = np.zeros((n, 3)); e = np.zeros(n, np.int32); t = np.zeros(n, np.int32)
        lib.emu_mesh_distance(h, x.ctypes.data_as(dp), n, signed, d.ctypes.data_as(dp), nr.ctypes.data_as(dp), e.ctypes.data_as(i32p), t.ctypes.data_as(i32p))
        total += n
        key = f"k1_fuzz/points/{seed}/{k}/signed={signed}"
        if not ref_check(key, (d, nr, e, t), lambda: RefMesh(V, F).distance(x, signed=bool(signed))):
            bad += 1
            print(f"MISMATCH {key} (kind {k % 7}, {len(F)} tris)")
    lib.emu_mesh_destroy(h)
print(f"{rounds} meshes, {total} queries, {bad} mismatches (result sets that differ from the reference)")
sys.exit(1 if bad else 0)
