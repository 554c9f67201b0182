#!/usr/bin/env python
"""Parity fuzzer (CPU) for interpolate: the product's K2 kernel code run by tests/emu (build/bin/libk23emu.so) against the reference's own
CubicLagrangeDiscreteGrid::interpolate (oracle/_ref/libdiscregrid_ref.so) on random grids (anisotropic, offset, tiny / huge cells), random
fields with DBL_MAX sentinels, optionally reduced, and queries that sit on cell faces, domain corners and outside, plus NaN / infinities:
value + gradient and value-only, bit for bit.  The reduced fields are made by the product's dg_reduce_field (host passes) and checked against
the reference's reduceField first.  The reference's results come from tests/golden/ref_digests.json where they are stored for a case
(oracle_api.ref_check), from oracle/_ref otherwise; a mismatch is reported per case.  usage: tools/k2_fuzz.py [rounds=60] [seed=0]"""
import ctypes as C, os, sys, tempfile
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from oracle_api import Oracle, RefGrid, ref_check
from make_reduce_golden import write_cdf
from test_oracle_golden import read_cdf
from test_reduce_field import reduce_field
import discregrid_b200 as dg
rounds = int(sys.argv[1]) if len(sys.argv) > 1 else 60
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
rng = np.random.default_rng(seed)
lib = C.CDLL(os.path.join(ROOT, "build", "bin", "libk23emu.so"))
dp, u32p = C.POINTER(C.c_double), C.POINTER(C.c_uint32)
lib.emu_field_create.restype = C.c_void_p
lib.emu_field_create.argtypes = [dp, u32p, dp, u32p, C.c_uint64, u32p]
lib.emu_field_destroy.argtypes = [C.c_void_p]
lib.emu_interpolate.argtypes = [C.c_void_p, dp, C.c_uint64, dp, dp]
orc = Oracle()
DBL_MAX = np.finfo(np.float64).max
tmp = tempfile.mkdtemp(dir=os.path.join(ROOT, "build"))
bad = total = 0
for k in range(rounds):
    res = tuple(int(v) for v in rng.integers(1, 7, 3))
    sc = 10.0 ** rng.integers(-5, 6)
    mn = rng.standard_normal(3) * sc * 10 ** rng.integers(0, 3)
    mx = mn + sc * (0.2 + rng.random(3) * (10 ** rng.integers(0, 2, 3)))
    gd, r = orc.grid_desc(mn, mx, res)
    cells = orc.build_cells(r)
    n = int(cells.max()) + 1
    v = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4)
    if k % 3 == 1: v[rng.random(n) < 0.05] = DBL_MAX                 # missing coefficients
    src, dst = os.path.join(tmp, "in.cdf"), os.path.join(tmp, "reduced.cdf")
    write_cdf(src, mn, mx, res, gd[6:9], gd[9:12], v, cells, np.arange(len(cells), dtype=np.uint32))
    g = read_cdf(src)
    field = (g["nodes"][0], g["cells"][0], g["cmap"][0])

    def ref_grid():
        ref = RefGrid(src)
        if k % 3 == 2:
            ref.reduce_window(0, lo, hi); ref.save(dst); ref.close(); ref = RefGrid(dst)
        return ref
    if k % 3 == 2:                                                    # a reduced field: removed cells, renumbered nodes
        lo, hi = float(np.quantile(v, 0.3)), float(np.quantile(v, 0.7))
        field = reduce_field(dg, g, v, (lo <= v) & (v <= hi) & (v != DBL_MAX), cells)

        def ref_reduced():
            ref_grid().close(); r_ = read_cdf(dst)
            return r_["nodes"][0], r_["cells"][0], r_["cmap"][0]
        if not ref_check(f"k2_fuzz/{seed}/{k}/reduced", field, ref_reduced, nan_equal=False):
            bad += 1
            print(f"MISMATCH k2_fuzz/{seed}/{k}/reduced: dg_reduce_field differs from the reference's reduceField")
    ext = mx - mn
    xs = [mn - 0.1 * ext + rng.random((400, 3)) * 1.2 * ext]
    faces = [mn[d] + gd[6 + d] * np.arange(res[d] + 1) for d in range(3)]
    xs.append(np.stack([rng.choice(faces[0], 200), rng.choice(faces[1], 200), rng.choice(faces[2], 200)], 1))                     # cell corners
    on_face = mn + rng.random((200, 3)) * ext; on_face[:, 0] = rng.choice(faces[0], 200); xs.append(on_face)                      # on x-faces
    xs.append(np.array([mn, mx, [mn[0], mx[1], mn[2]], 0.5 * (mn + mx), np.nextafter(mx, np.inf), np.nextafter(mn, -np.inf),
                        [np.nan, mn[1], mn[2]], [np.inf, mn[1], mn[2]], [mn[0], -np.inf, mn[2]], [0.0, 0.0, 0.0], [-0.0, -0.0, -0.0]]))
    x = np.ascontiguousarray(np.concatenate(xs)); m = len(x)

    def ref_interpolate():
        ref = ref_grid()
        want = ref.interpolate(0, x, grad=True) + (ref.interpolate(0, x, grad=False)[0],)
        ref.close()
        return want
    nodes = np.ascontiguousarray(field[0]); cc = np.ascontiguousarray(field[1], np.uint32); cm = np.ascontiguousarray(field[2], np.uint32)
    h = lib.emu_field_create(gd.ctypes.data_as(dp), r.ctypes.data_as(u32p), nodes.ctypes.data_as(dp), cc.ctypes.data_as(u32p), len(cc), cm.ctypes.data_as(u32p))
    phi = np.zeros(m); grad = np.zeros((m, 3)); only = np.zeros(m)
    lib.emu_interpolate(h, x.ctypes.data_as(dp), m, phi.ctypes.data_as(dp), grad.ctypes.data_as(dp))
    lib.emu_interpolate(h, x.ctypes.data_as(dp), m, only.ctypes.data_as(dp), None)
    lib.emu_field_destroy(h)
    total += m
    if not ref_check(f"k2_fuzz/{seed}/{k}", (phi, grad, only), ref_interpolate):
        bad += 1
        print(f"MISMATCH k2_fuzz/{seed}/{k} res {res}")
print(f"{rounds} fields, {total} queries, {bad} mismatches (result sets that differ from the reference)")
sys.exit(1 if bad else 0)
