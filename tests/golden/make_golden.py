"""Regenerates the committed golden fixtures.  Run where the reference is compiled: `make -C oracle ref REF=<checkout of the
reference>` builds oracle/_ref (libdgref.so = its own unmodified TriangleMeshDistance.h, its grid class and tools) and stages its meshes:

    python tests/golden/make_golden.py

Outputs (all small, committed):
  box.obj, box.cdf           verbatim copies of the reference's only golden vector
                             (cmd/generate_sdf/resources/box.{obj,cdf}; box.cdf = GenerateSDF -r "5 5 5" box.obj)
  ref_torus_queries.npz      reference-header results (distance, nearest point, entity, triangle) for 4000 seeded
                             points around a deterministic 4,608-triangle bumpy torus (discregrid_b200.mesh.bumpy_torus)
  ref_torus_tree.npz         the reference's tree (children + internal spheres) and pseudonormals for that torus
  ref_sphere_surface.npz     reference results for points ON / very near a UV sphere's surface (ties, sign near 0)
  ref_digests.json           sha256 digests of the reference's results where the arrays would be too large to commit
                             (oracle_api.ref_check): the tests that compare with the reference on generated inputs are run
                             with DG_RECORD_REF_DIGESTS=1 at the end of this script
"""
import json, os, shutil, sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle_api import REF_DIGESTS, REF_RESOURCES as REF_RES, RefMesh, Oracle, digest   # noqa: E402
import ctypes as C                             # noqa: E402
from discregrid_b200.mesh import bumpy_torus, uv_sphere   # noqa: E402 (pure numpy part of the package)

for f in ("box.obj", "box.cdf"):
    shutil.copyfile(os.path.join(REF_RES, f), os.path.join(HERE, f))
    os.chmod(os.path.join(HERE, f), 0o644)

orc = Oracle()
torus = bumpy_torus(48, 48, 1.0, 0.4, 0.05, 7, 5)            # 4608 triangles
ref = RefMesh(torus.vertices, torus.faces)
mn, mx = orc.generate_sdf_domain(torus.vertices)
rng = np.random.default_rng(20260924)
x = mn + rng.random((4000, 3)) * (mx - mn)
d, near, ent, tri = ref.distance(x, signed=True)
du = ref.distance(x, signed=False)[0]
np.savez_compressed(os.path.join(HERE, "ref_torus_queries.npz"), x=x, distance=d, unsigned=du, nearest=near,
                    entity=ent, triangle=tri, torus_args=np.array([48, 48, 1.0, 0.4, 0.05, 7, 5]))
sph, kids = ref.tree()
pt, pe, pv = ref.pseudonormals()
internal = kids[:, 0] != -1
np.savez_compressed(os.path.join(HERE, "ref_torus_tree.npz"), kids=kids, spheres_internal=sph[internal], pn_tri=pt, pn_edge=pe, pn_vert=pv)

s = uv_sphere(12, 24, 0.75, (0.1, -0.2, 0.05))
refs = RefMesh(s.vertices, s.faces)
V, F = s.vertices, s.faces
pts = [V.copy()]                                             # exactly on vertices
pts.append(0.5 * (V[F[:, 0]] + V[F[:, 1]]))                  # on edge midpoints
pts.append((V[F[:, 0]] + V[F[:, 1]] + V[F[:, 2]]) / 3.0)     # face centroids
c = (V[F[:, 0]] + V[F[:, 1]] + V[F[:, 2]]) / 3.0
pts.append(c * (1 + 1e-9)); pts.append(c * (1 - 1e-9)); pts.append(V * (1 + 1e-12))
xs = np.concatenate(pts, 0)
d, near, ent, tri = refs.distance(xs, signed=True)
np.savez_compressed(os.path.join(HERE, "ref_sphere_surface.npz"), x=xs, distance=d, nearest=near, entity=ent, triangle=tri,
                    sphere_args=np.array([12, 24, 0.75, 0.1, -0.2, 0.05]))

# ---------------------------------------------------------------------------------------------------------------------
# Fixtures produced by the reference's OWN tools and grid class (unmodified sources compiled against the Eigen stand-in
# oracle/ref_eigen; `make -C oracle ref`).  First the build is validated: its GenerateSDF must reproduce box.cdf byte for byte.
import subprocess, tempfile
from oracle_api import REF_BIN, RefGrid
tmp = tempfile.mkdtemp()
run = lambda *a: subprocess.run(list(a), check=True, capture_output=True)
run(os.path.join(REF_BIN, "GenerateSDF"), "-r", "5 5 5", "-o", os.path.join(tmp, "box.cdf"), os.path.join(HERE, "box.obj"))
assert open(os.path.join(tmp, "box.cdf"), "rb").read() == open(os.path.join(HERE, "box.cdf"), "rb").read(), "stand-in build does not reproduce box.cdf"

sph = uv_sphere(10, 16, 0.5)
sph.exportOBJ(os.path.join(HERE, "sphere.obj"))
run(os.path.join(REF_BIN, "GenerateSDF"), "-r", "10 10 10", "-d", "-2 -2 -2 2 2 2", "-o", os.path.join(HERE, "ref_sphere.cdf"), os.path.join(HERE, "sphere.obj"))
run(os.path.join(REF_BIN, "GenerateSDF"), "-i", "-r", "4 6 5", "-o", os.path.join(HERE, "ref_sphere_inverted_padded.cdf"), os.path.join(HERE, "sphere.obj"))
run(os.path.join(REF_BIN, "GenerateDensityMap"), "-s", "0.15", "-r", "1000", "--no-reduction", "-o", os.path.join(HERE, "ref_sphere_noreduction.cdm"),
    os.path.join(HERE, "ref_sphere.cdf"))
run(os.path.join(REF_BIN, "GenerateDensityMap"), "-s", "0.15", "-r", "1000", "-o", os.path.join(HERE, "ref_sphere_reduced.cdm"), os.path.join(HERE, "ref_sphere.cdf"))
run(os.path.join(REF_BIN, "DiscreteFieldToBitmap"), "-s", "64", "-p", "xz", "-d", "0.25", "-o", os.path.join(HERE, "ref_box_xz.bmp"), os.path.join(HERE, "box.cdf"))
run(os.path.join(REF_BIN, "DiscreteFieldToBitmap"), "-s", "48", "-p", "yx", "-f", "1", "-c", "rs", "-o", os.path.join(HERE, "ref_sphere_density_yx.bmp"),
    os.path.join(HERE, "ref_sphere_noreduction.cdm"))

# a real mesh end to end through the reference tool (the mesh itself is not committed: GPU-side tests find it under oracle/_ref/resources)
run(os.path.join(REF_BIN, "GenerateSDF"), "-r", "12 12 12", "-o", os.path.join(HERE, "ref_bunny_12.cdf"), os.path.join(REF_RES, "bunny.obj"))
run(os.path.join(REF_BIN, "GenerateSDF"), "-i", "-r", "10 10 10", "-o", os.path.join(HERE, "ref_dragon_10_inverted.cdf"), os.path.join(REF_RES, "dragon.obj"))
# 855,196 triangles, not watertight (edges with more than two triangles): the sign follows whatever pseudonormals that gives
run(os.path.join(REF_BIN, "GenerateSDF"), "-r", "8 8 8", "-o", os.path.join(HERE, "ref_buddha_8.cdf"), os.path.join(REF_RES, "happy_buddha.obj"))

rng = np.random.default_rng(77)
out = {}
for tag, path, fields in (("box", "box.cdf", (0,)), ("red", "ref_sphere_reduced.cdm", (0, 1)), ("nr", "ref_sphere_noreduction.cdm", (1,))):
    g = RefGrid(os.path.join(HERE, path))
    dom = np.empty(6); res = np.empty(3, np.uint32); cell = np.empty(3); inv = np.empty(3); nc = C.c_uint64()
    import ctypes as C2
    g.lib.refg_info.argtypes = [C2.c_void_p, C2.POINTER(C2.c_double), C2.POINTER(C2.c_uint32), C2.POINTER(C2.c_double), C2.POINTER(C2.c_double), C2.POINTER(C2.c_uint64)]
    nc = C2.c_uint64()
    g.lib.refg_info(g.h, dom.ctypes.data_as(C2.POINTER(C2.c_double)), res.ctypes.data_as(C2.POINTER(C2.c_uint32)), cell.ctypes.data_as(C2.POINTER(C2.c_double)),
                    inv.ctypes.data_as(C2.POINTER(C2.c_double)), C2.byref(nc))
    lo, hi = dom[:3], dom[3:]
    xq = lo - 0.03 * (hi - lo) + rng.random((6000, 3)) * 1.06 * (hi - lo)
    xq[:4] = [lo, hi, 0.5 * (lo + hi), [hi[0], lo[1], hi[2]]]
    out[tag + "_x"] = xq
    for f in fields:
        phi, grad = g.interpolate(f, xq, grad=True)
        out[f"{tag}_f{f}_phi"], out[f"{tag}_f{f}_grad"] = phi, grad
        out[f"{tag}_f{f}_phi_only"] = g.interpolate(f, xq, grad=False)[0]
    if tag == "box":
        ok, N, dN, c0, cells, phi2, grad2 = g.split(0, xq[:1500])
        out.update(box_split_ok=ok, box_split_c0=c0, box_split_cell=cells, box_split_phi=phi2, box_split_grad=grad2)
        # the shape functions and their gradients (1500 x 32 x 4 doubles) would take the file past 1 MB: kept as a digest
        digests = json.load(open(REF_DIGESTS)) if os.path.exists(REF_DIGESTS) else {}
        digests["ref_grid_queries/box_split_N_dN"] = digest((N[ok.astype(bool)], dN[ok.astype(bool)]), nan_equal=False)
        with open(REF_DIGESTS, "w") as f:
            json.dump(digests, f, indent=0, sort_keys=True)
            f.write("\n")
np.savez_compressed(os.path.join(HERE, "ref_grid_queries.npz"), **out)

# reduceField on an ANISOTROPIC grid: cells of 1/6 x 1/3 x 2/3 make several surviving nodes share one Morton key (the key's cell
# size is the largest one, :1114), so the node order of the result depends on how std::sort leaves equal keys -- the case
# dg_reduce_field handles by replaying the reference's own sort.  Input and the reference's output are both committed.
subprocess.run([sys.executable, os.path.join(HERE, "make_reduce_golden.py")], check=True)

# digests of the reference's results on the inputs the tests generate (oracle_api.ref_check): the tests record them themselves
subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-m", "not gpu", "-k",
                "awkward or non_finite or fuzz or against_the_reference_library or real_addfunction",
                "tests/test_k1_emulated.py", "tests/test_k23_emulated.py", "tests/test_reduce_field.py", "tests/test_oracle_reference_tools.py"],
               cwd=ROOT, env=dict(os.environ, DG_RECORD_REF_DIGESTS="1"), check=True)
print("golden fixtures written to", HERE)
