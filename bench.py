#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Discregrid hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): "SDF grid nodes/sec (addFunction) + interpolate Mqueries/sec".
Workload at N = 1: BASELINE.json configs[1], "Stanford bunny (~70k tris) 128^3 grid, 1xB200, fp64" -- the reference's own bunny.obj
(69,630 triangles; staged as an INPUT file under oracle/_ref/resources by `make -C oracle ref`, it travels to the GPU box) on the
GenerateSDF-padded domain; when the file is not staged, a synthetic closed mesh of the same size (69,564 triangles) and the line says so.
A "step" = one full pass of the addFunction node loop over the 14,926,977 nodes.

  value      nodes/s of the node loop, coefficients device-resident (CUDA events, max over ranks)
  e2e        the same metric through the C-ABI call a caller makes, dg_add_function_sdf(mesh, grid, sign, nodes, cells, cell_map):
             the WHOLE of CubicLagrangeDiscreteGrid::addFunction (cubic_lagrange_discrete_grid.cpp:780-899) -- node loop, D2H of the
             coefficient array, 32-index connectivity table, cell map -- into freshly allocated host arrays, wall-clock
  roofline   K1 against the measured fp64 issue rate (dg_fp64_rate_probe: DMUL+DADD, no FMA -- the numerical contract), with the HBM
             view and the interpolate kernel's HBM roofline nested
  cpu_baseline / --impl reference
             the reference's REAL addFunction (oracle/_ref/libdiscregrid_ref.so = its unmodified sources, oracle/ref_grid_wrapper.cpp:
             refg_add_function_sdf) with the GenerateSDF functor on the host cores, whole grid, timed around the call exactly as e2e is.
             Threads: all logical CPUs of the affinity mask, or 2 x the cgroup CPU quota when one is in force (the measured optimum on
             both kinds of box), OMP_PROC_BIND=spread OMP_PLACES=threads.  The CPU work always runs in a child process so that these
             settings are in place before libgomp starts; the line reports cores, quota and the per-thread rate so that runs on
             differently provisioned hosts can be compared.
The second half of the metric, interpolate()+gradient Mqueries/s (config 4: 10 M uniform random queries on a 256^3 SDF), is carried
under "interpolate" and nested in roofline / e2e / cpu_baseline (the driver keeps those objects whole).
"""
import argparse
import atexit
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # the benchmark writes nothing into the source tree (no __pycache__ either)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = {"source": "bunny", "resolution": [128, 128, 128], "torus": (186, 187, 1.0, 0.4, 0.05, 7, 5)}
INTERP = {"resolution": [256, 256, 256], "queries": 10_000_000, "seed": 0x5EED}
# --dump-outputs: 2^21 of the headline grid's nodes (16 MB) and 2^20 of the interpolate queries (phi + gradient, 32 MB)
DUMP = {"sdf_nodes": 1 << 21, "queries": 1 << 20, "seed": 0xD1F}
# the reference's meshes (inputs), staged by `make -C oracle ref`; DG_BENCH_MESH_DIR points elsewhere (the CPU rehearsal stages small stand-ins)
RES_DIR = os.environ.get("DG_BENCH_MESH_DIR") or os.path.join(ROOT, "oracle", "_ref", "resources")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--resolution", type=int, default=0, help="override the SDF grid resolution (diagnostics)")
    ap.add_argument("--interp-resolution", type=int, default=0, help="override the interpolate grid resolution (diagnostics)")
    ap.add_argument("--target-resolution", type=int, default=256, help="grid resolution of the target-config leg (diagnostics / rehearsal; the config is 256)")
    ap.add_argument("--real-resolution", type=int, default=0, help="override the grid resolution of the reference-mesh leg (diagnostics / rehearsal)")
    ap.add_argument("--mesh", default="", choices=["", "bunny", "torus"], help="override the headline mesh (default: bunny.obj when staged, else the synthetic torus)")
    ap.add_argument("--no-interp", action="store_true", help="skip the interpolate half (diagnostics / profiling)")
    ap.add_argument("--no-cpu", action="store_true", help="skip every CPU leg (diagnostics / profiling)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the e2e leg (diagnostics / profiling)")
    ap.add_argument("--no-target", action="store_true", help="skip the 256^3 / 100k-triangle target-config leg")
    ap.add_argument("--sharding", default="auto", choices=["auto", "slab", "chunks", "interleaved"],
                    help="N>1: round-robin node-id chunks, whole-plane slabs, or plane pairs dealt round-robin (one launch + one all-gather + unpack); "
                         "auto = interleaved from 4 ranks up, chunks below")
    ap.add_argument("--splits", type=int, default=1, help="interleaved sharding: launches per rank (each on its own stream; world * splits <= 16)")
    ap.add_argument("--no-real", action="store_true", help="skip the leg on the other reference meshes (dragon / happy_buddha)")
    ap.add_argument("--no-density", action="store_true", help="skip the density-map (K3) legs (diagnostics / profiling)")
    ap.add_argument("--cpu-seconds", type=float, default=40.0, help="a CPU leg whose full-size run is estimated to take longer than this falls back to a strided sample")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what they computed as DIR/<name>.npy (float64; fixed seeded samples of the large arrays)")
    ap.add_argument("--cpu-child", default="", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.sharding == "auto":
        args.sharding = "interleaved" if int(os.environ.get("WORLD_SIZE", "1")) >= 4 else "chunks"
    return args


# ------------------------------------------------------------------------------------------------ helpers
_SCRATCH = []


def scratch_dir():
    """for the few hundred MB some legs exchange through files: a private temporary directory, removed at exit (the source tree may be
    read-only, and the benchmark leaves nothing in it)"""
    if not _SCRATCH:
        _SCRATCH.append(tempfile.mkdtemp(prefix="dg_bench_"))
        atexit.register(shutil.rmtree, _SCRATCH[0], True)
    return _SCRATCH[0]


def dump_sample(n, k, seed):
    """--dump-outputs: a fixed, seeded, sorted sample of k of the indices 0..n-1 (all of them when n <= k)"""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def dump_outputs(path, arrays):
    """--dump-outputs: every array as <path>/<name>.npy in float64"""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float64))


def workload_mesh(dg, source, torus=None):
    """-> (mesh, description, data tag).  'bunny' = the reference's bunny.obj when staged."""
    if source in ("bunny", "dragon", "happy_buddha"):
        p = os.path.join(RES_DIR, source + ".obj")
        if os.path.exists(p):
            m = dg.TriangleMesh(p)
            return m, f"{source}.obj of the reference ({m.nFaces()} triangles / {len(m.vertices)} vertices)", "reference mesh file"
        source = "torus"
    if source == "target":
        m = dg.bumpy_torus()
        return m, "synthetic bumpy torus, 250x200 quads = exactly 100,000 triangles / 50,000 vertices (BASELINE.md target config)", "synthetic"
    m = dg.bumpy_torus(*(torus or WORKLOAD["torus"]))
    return m, f"synthetic bumpy torus, {m.nFaces()} triangles / {len(m.vertices)} vertices (bunny-class: bunny.obj has 69,630; the file is not staged here)", "synthetic"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md 6.65 TB/s)"


def splitmix_points(n, seed, lo, hi):
    """BASELINE.md config 4: u = (splitmix64(seed, counter = 3q + d) >> 11) * 2^-53, x_d = lo_d + u * (hi_d - lo_d)."""
    with np.errstate(over="ignore"):
        z = (np.uint64(seed) + (np.arange(3 * n, dtype=np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u = (z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    return lo + u.reshape(n, 3) * (hi - lo)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_policy():
    """Host threads for the reference's OpenMP loops: every logical CPU of the affinity mask -- the BVH walk is latency-bound and gains from
    SMT (measured on the B200 hosts: 128 threads on 64 cores 13.0 vs 9.8 Mnodes/s with 64) -- unless a cgroup CPU quota is in force: a 1-GPU
    lease of this pool sees 128 logical CPUs under `cpu.max = 16 CPUs`, where 128 busy threads are SLOWER than 32 (1.85 vs 2.09 Mnodes/s,
    profiles/r2a_cpuarm.txt); then 2 x quota threads.  Threads are spread and pinned (OMP_PROC_BIND=spread, OMP_PLACES=threads).
    DG_CPU_THREADS overrides the count."""
    allowed = sorted(os.sched_getaffinity(0))
    cores = {}
    for c in allowed:
        try:
            sib = open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read().strip()
        except OSError:
            sib = str(c)
        cores.setdefault(sib, c)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except (OSError, ValueError):
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and per > 0:
                quota = q / per
        except (OSError, ValueError):
            pass
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    threads = len(allowed) or 1
    if quota is not None and quota >= 1:
        threads = max(1, min(threads, int(2 * quota)))
    if os.environ.get("DG_CPU_THREADS"):
        threads = int(os.environ["DG_CPU_THREADS"])
    env = {"OMP_NUM_THREADS": str(threads), "OMP_PROC_BIND": os.environ.get("DG_OMP_PROC_BIND", "spread"),
           "OMP_PLACES": os.environ.get("DG_OMP_PLACES", "threads"), "OMP_DYNAMIC": "false"}
    return {"threads": threads, "logical_cpus": len(allowed), "physical_cores": len(cores), "cgroup_cpu_quota": quota, "cpu_model": model, "omp_env": env}


def run_cpu_child(spec, timeout=1800):
    """Runs one CPU leg in a child process whose OpenMP environment is set before libgomp starts.  -> result dict (or {"error": ...})"""
    pol = cpu_policy()
    env = dict(os.environ, **pol["omp_env"])
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_RUN_ID"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-child", json.dumps(spec)], capture_output=True, text=True, env=env, timeout=timeout)
    except subprocess.TimeoutExpired:
        return {"error": f"cpu child timed out after {timeout} s"}
    for line in reversed(r.stdout.splitlines()):
        if line.startswith('{"cpu_child"'):
            d = json.loads(line)
            d.pop("cpu_child")
            d.update({k: pol[k] for k in ("logical_cpus", "physical_cores", "cgroup_cpu_quota", "cpu_model")})
            d["omp"] = {k: v for k, v in pol["omp_env"].items() if k != "OMP_DYNAMIC"}
            return d
    return {"error": f"cpu child rc={r.returncode}: {(r.stdout + r.stderr)[-600:]}"}


def _child_mesh(spec):
    import discregrid_b200 as dg
    return workload_mesh(dg, spec["mesh"], spec.get("torus"))[0]


def cpu_child_addfunction(spec):
    """The reference's real addFunction on the whole grid, `runs` times (+ `warm` untimed), optionally checked against the GPU result."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import discregrid_b200 as dg
    from oracle_api import Oracle, RefAddFunction, RefMesh, have_ref, have_ref_grid
    mesh = _child_mesh(spec)
    mn, mx = dg.generate_sdf_domain(mesh.vertices)
    res = spec["res"]
    orc = Oracle()
    gd, r = orc.grid_desc(mn, mx, res)
    n_nodes = orc.num_nodes(r)
    threads = int(os.environ.get("OMP_NUM_THREADS", "0")) or orc.max_threads()
    out = {"n_nodes": n_nodes, "cores": threads}
    # traversal statistics of the reference algorithm on a strided node sample (single-threaded counters of the oracle port): the
    # algorithmic flop count of K1's roofline, SURVEY 8(d): visits * 24 + leaf tests * 65
    if spec.get("stats_nodes"):
        ids = np.linspace(0, n_nodes - 1, int(spec["stats_nodes"])).astype(np.int64)
        v, l = orc.mesh(mesh.vertices, mesh.faces).stats(orc.node_positions_at(gd, r, ids))
        out.update(visits_per_node=v, leaf_tests_per_node=l, flops_per_node=24.0 * v + 65.0 * l)
    # calibration on 20k strided nodes with the reference's signed_distance: is the full-size call affordable?
    est = None
    if have_ref():
        rm = RefMesh(mesh.vertices, mesh.faces)
        ids = np.linspace(0, n_nodes - 1, 20_000).astype(np.int64)
        x = orc.node_positions_at(gd, r, ids)
        rm.sample_points(x[:2000], nthreads=threads)
        t0 = time.perf_counter(); rm.sample_points(x, nthreads=threads); dt = time.perf_counter() - t0
        est = dt / len(ids) * n_nodes
        out["calibration_nodes_per_s"] = len(ids) / dt
    runs, warm = int(spec.get("runs", 1)), int(spec.get("warm", 0))
    full = have_ref_grid() and (est is None or est * (runs + warm) <= float(spec.get("max_seconds", 60.0)))
    if full:
        ref = RefAddFunction(mesh.vertices, mesh.faces)
        times, nodes, cells = [], None, None
        want = bool(spec.get("check_gpu"))
        for it in range(warm + runs):
            last = it == warm + runs - 1
            dt, nn, cc = ref.add_function(mn, mx, res, nthreads=threads, want_nodes=want and last, want_cells=want and last and n_nodes < 40_000_000)
            if it >= warm:
                times.append(dt)
            if last:
                nodes, cells = nn, cc
        out.update(kind="reference", mode="full_addfunction", times_s=times,
                   sample=f"the reference's real CubicLagrangeDiscreteGrid::addFunction(GenerateSDF functor, verbose=false) over all {n_nodes} nodes "
                          f"({runs} timed call(s) after {warm} warm-up), node loop + connectivity + cell map, steady_clock around the call")
        if want:
            # full-size parity, by-product of the baseline: every node (and every cell index) the reference produced vs the GPU path
            md = dg.TriangleMeshDistance(mesh)
            g = dg.CubicLagrangeDiscreteGrid(mn, mx, res)
            g.addFunction(dg.MeshSignedDistance(md))
            out["parity_nodes_bit_exact"] = bool(np.array_equal(g.m_nodes[0].view(np.uint64), nodes.view(np.uint64)))
            out["parity_nodes_compared"] = int(n_nodes)
            if cells is not None:
                out["parity_cells_equal"] = bool(np.array_equal(g.m_cells[0], cells))
    else:
        # bounded sample: the node-loop body on evenly strided nodes (positions by the oracle's indexToNodePosition, untimed)
        kind = "reference" if have_ref() else "port"
        m = RefMesh(mesh.vertices, mesh.faces) if kind == "reference" else orc.mesh(mesh.vertices, mesh.faces)
        budget = float(spec.get("max_seconds", 60.0)) / max(1, runs + warm)
        n_sample = int(min(n_nodes, max(20_000, (budget / est * n_nodes) if est else 200_000)))
        ids = np.linspace(0, n_nodes - 1, n_sample).astype(np.int64)
        x = orc.node_positions_at(gd, r, ids)
        times = []
        for it in range(warm + runs):
            t0 = time.perf_counter()
            if kind == "reference":
                m.sample_points(x, nthreads=threads)
            else:
                m.distance(x)
            if it >= warm:
                times.append((time.perf_counter() - t0) * n_nodes / n_sample)           # scaled to the full grid
        out.update(kind=kind, mode="strided_sample", times_s=times,
                   sample=f"{n_sample} of {n_nodes} nodes, evenly strided, OpenMP schedule(static), node-loop body only "
                          f"({'reference TriangleMeshDistance.h' if kind == 'reference' else 'oracle port'}); times scaled to the full grid "
                          f"(the full call was estimated at {est:.1f} s per run)" if est else "strided sample")
    return out


def cpu_child_interp(spec):
    """The reference's own CubicLagrangeDiscreteGrid::interpolate(field, x, &grad) in the OpenMP loop of cmd/discrete_field_to_bitmap/main.cpp:118-135
    over the SAME queries on the SAME field as the GPU leg; the field is built on the GPU (input preparation), the grid object by the reference's
    own addFunction, and every query's value + gradient is compared with the GPU's."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import discregrid_b200 as dg
    from oracle_api import Oracle, RefGridInMemory, have_ref_grid
    mesh = _child_mesh(spec)
    mn, mx = dg.generate_sdf_domain(mesh.vertices)
    res, nq = spec["res"], int(spec["queries"])
    md = dg.TriangleMeshDistance(mesh)
    g = dg.CubicLagrangeDiscreteGrid(mn, mx, res)
    g.addFunction(dg.MeshSignedDistance(md))
    x = np.ascontiguousarray(splitmix_points(nq, spec["seed"], mn, mx))
    pg, gg = g.interpolate(0, x, gradient=True)
    threads = int(os.environ.get("OMP_NUM_THREADS", "0"))
    out = {"queries": nq, "cores": threads}
    if have_ref_grid():
        rg = RefGridInMemory(mn, mx, res, g.m_nodes[0], nthreads=threads)
        rg.interpolate(0, x[:200_000], grad=True, nthreads=threads)
        best = None
        for _ in range(int(spec.get("runs", 2))):
            t0 = time.perf_counter(); pr, gr = rg.interpolate(0, x, grad=True, nthreads=threads); dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        out.update(kind="reference", seconds=best,
                   sample=f"all {nq} queries on the {res[0]}^3 field ({len(g.m_nodes[0])} nodes): the reference class's interpolate(0, x, &grad) in an OpenMP parallel for, best of {spec.get('runs', 2)}")
    else:
        orc = Oracle(); gd, r = orc.grid_desc(mn, mx, res)
        t0 = time.perf_counter(); pr, gr = orc.interpolate(gd, r, g.m_nodes[0], x, grad=True); best = time.perf_counter() - t0
        out.update(kind="port", seconds=best, sample=f"all {nq} queries on the {res[0]}^3 field, oracle port")
    out["bit_exact_vs_gpu"] = bool(np.array_equal(pr.view(np.uint64), pg.view(np.uint64)) and np.array_equal(gr.view(np.uint64), gg.view(np.uint64)))
    out["queries_compared"] = nq
    return out


def cpu_child_main(spec):
    fn = {"addfunction": cpu_child_addfunction, "interp": cpu_child_interp}[spec["what"]]
    out = fn(spec)
    out["cpu_child"] = 1
    # key order: the parent looks for a line starting with {"cpu_child"
    print(json.dumps({"cpu_child": 1, **{k: v for k, v in out.items() if k != "cpu_child"}}))


def addfunction_baseline(source, torus, res, runs, warm, max_seconds, check_gpu, stats_nodes=4000):
    d = run_cpu_child({"what": "addfunction", "mesh": source, "torus": torus, "res": list(res), "runs": runs, "warm": warm,
                       "max_seconds": max_seconds, "check_gpu": check_gpu, "stats_nodes": stats_nodes})
    if "error" in d:
        return d
    t = d["times_s"]
    d["value"] = d["n_nodes"] / float(np.mean(t)); d["unit"] = "nodes/s"; d["best_value"] = d["n_nodes"] / min(t)
    d["value_per_thread"] = d["value"] / max(1, d["cores"])          # hosts of this pool differ in the CPUs a lease may use (16-CPU quota vs 128)
    return d


# ------------------------------------------------------------------------------------------------ main
def main():
    args = parse()
    if args.cpu_child:
        cpu_child_main(json.loads(args.cpu_child))
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    res = [args.resolution] * 3 if args.resolution else WORKLOAD["resolution"]
    source = args.mesh or WORKLOAD["source"]

    import discregrid_b200 as dg           # fails loudly if the CUDA library is not built
    from discregrid_b200 import _capi as capi

    mesh, mesh_text, data_tag = workload_mesh(dg, source)
    if data_tag == "synthetic":
        source = "torus"
    mn, mx = dg.generate_sdf_domain(mesh.vertices)
    desc = dg.grid_desc(mn, mx, res)
    n_nodes = C.c_uint64()
    capi.check(capi.lib.dg_grid_num_nodes(desc.resolution, C.byref(n_nodes)))
    n_nodes = n_nodes.value
    n_cells = int(res[0]) * int(res[1]) * int(res[2])
    par = f"x{world}" + ("" if world == 1 else (", slabs of whole plane pairs of the four node arrays: one launch per rank + one NCCL all-gather per node array" if args.sharding == "slab" else ", plane pairs dealt round-robin: one launch per rank + ONE NCCL all-gather + unpack kernel" if args.sharding == "interleaved" else ", 2 round-robin node-id chunks per rank on 2 streams + one in-place NCCL all-gather per row"))
    config = {"workload": f"GenerateSDF addFunction (BASELINE.json configs[1]): {mesh_text}; {res[0]}x{res[1]}x{res[2]} grid = {n_nodes} nodes; "
                          "GenerateSDF-padded domain; fp64 bit-exact with the reference",
              "mesh_triangles": int(mesh.nFaces()), "grid": res, "nodes": n_nodes,
              "l2": "flushed between timed iterations (256 MiB write)", "parallelism": par}
    data = f"{data_tag} + regular grid" if data_tag != "synthetic" else "synthetic"

    # ---------------------------------------------------------------- reference arm (CPU): the reference's real addFunction per step
    if args.impl == "reference":
        if rank != 0:
            return
        d = addfunction_baseline(source, WORKLOAD["torus"], res, runs=args.steps, warm=min(args.warmup, 1), max_seconds=args.cpu_seconds * 6, check_gpu=False, stats_nodes=0)
        if "error" in d:
            print(json.dumps({"impl": "reference", "unavailable": d["error"][:300]}))
            return
        v = d["value"]
        line = {"impl": "reference", "metric": "SDF grid nodes/sec (addFunction)", "value": v, "unit": "nodes/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * n_nodes / v, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": data, "config": config,
                "cpu_baseline": {k: d[k] for k in d if k not in ("times_s",)},
                "e2e": {"value": v, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
                "timing": {"per_step_s": d["times_s"], "best_value": d["best_value"]}}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- our arm (GPU)
    import torch
    import torch.distributed as dist
    from discregrid_b200.distributed import make_sharding, ShardedSdfSampler, SlabSdfSampler, InterleavedSdfSampler
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    assert not hasattr(capi.lib, "emu_mesh_create") or os.environ.get("DG_ALLOW_EMULATED_LIBRARY") == "1", "bench.py must run on the CUDA build of the library"
    torch.cuda.set_device(local_rank)
    capi.check(capi.lib.dg_set_device(local_rank))
    if world > 1:
        # NCCL_DEBUG stays unset: WARN would make NCCL print its version banner on stdout, next to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # a host-side group: ranks that must stay OFF their GPU (while rank 0 drives all GPUs from one process) wait in a gloo barrier -- an NCCL
    # barrier is a spinning kernel, and two processes on one GPU are time-sliced, which halves the throughput of the GPU being measured
    cpu_group = dist.new_group(backend="gloo") if world > 1 else None
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    md = dg.TriangleMeshDistance(mesh)
    mesh_info = md.info()
    sh = make_sharding(n_nodes, world)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    my_chunks = [(j, b, e) for (j, b, e) in sh.chunks_of(rank)]
    stream = torch.cuda.current_stream()

    def make_sampler(md_, desc_, n_):
        if args.sharding == "slab":
            return SlabSdfSampler(md_, desc_, rank, world)
        if args.sharding == "interleaved":
            return InterleavedSdfSampler(md_, desc_, rank, world, splits=args.splits if world * args.splits <= 16 else 1)
        return ShardedSdfSampler(md_, desc_, make_sharding(n_, world), rank)

    sdf_sampler = make_sampler(md, desc, n_nodes)
    full = torch.empty(sdf_sampler.sh.padded, dtype=torch.float64, device=dev)

    def same_as_single_launch(md_, desc_, n_, sharded):
        """every rank: the assembled array of the sharded step vs ONE dg_sample_sdf_device launch over all nodes on this GPU (bit-for-bit)"""
        if world == 1:
            return None
        single = torch.empty(n_, dtype=torch.float64, device=dev)
        capi.check(capi.lib.dg_sample_sdf_device(md_.handle, C.byref(desc_), 1.0, 0, n_, C.c_void_p(single.data_ptr()), C.c_void_p(stream.cuda_stream)))
        ok = bool(torch.equal(single.view(torch.int64), sharded[:n_].view(torch.int64)))
        del single
        return bool(max_over_ranks(0.0 if ok else 1.0) == 0.0)

    def timed(step_fn, steps, warmup):
        for _ in range(warmup):
            step_fn()
        times = []
        barrier()
        wall0 = time.perf_counter()
        for _ in range(steps):
            flush.fill_(1)                                  # L2 flush, outside the event pair
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); step_fn(); e1.record()
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        barrier()
        wall = time.perf_counter() - wall0
        return [max_over_ranks(t) for t in times], wall

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = dg.kernel_launch_count()
    sdf_ms, sdf_wall = timed(lambda: sdf_sampler.step(full), args.steps, args.warmup)
    launches = (dg.kernel_launch_count() - launches0) * args.steps // (args.steps + args.warmup)
    sharded_ok = same_as_single_launch(md, desc, n_nodes, full)
    clocks = sampler.stop() if rank == 0 else None
    dumped = {}
    if args.dump_outputs and rank == 0:
        # the coefficients of the last timed step, before any later leg reuses `full`
        idx = torch.from_numpy(dump_sample(n_nodes, DUMP["sdf_nodes"], DUMP["seed"])).to(dev)
        dumped["sdf_nodes"] = full[idx].cpu().numpy()
        del idx
    ms_step = float(np.mean(sdf_ms))
    value = n_nodes / (ms_step * 1e-3)

    # kernel-only time of K1 on this rank (no collective): what the roofline object refers to
    k1_ms, _ = timed(lambda: sdf_sampler.launch(full), max(3, args.steps // 2), 1)
    k1_ms = float(np.mean(k1_ms))
    if args.sharding == "slab" and world > 1:
        my_nodes = sum(e - b for (b, e) in sdf_sampler.sh.ranges[rank]); n_launch = 1
    elif args.sharding == "interleaved" and world > 1:
        my_nodes = n_nodes // world; n_launch = max(1, args.splits)
    else:
        my_nodes = sum(e - b for (_j, b, e) in my_chunks); n_launch = sum(1 for (_j, b, e) in my_chunks if e > b)
    peaks, peak_src = measured_peaks()
    fp64_peak = C.c_double()
    capi.check(capi.lib.dg_fp64_rate_probe(C.byref(fp64_peak)))
    fp64_peak = fp64_peak.value

    # ---------------------------------------------------------------- e2e: the whole addFunction through the C-ABI, HOST arrays
    e2e = None
    if not args.no_e2e:
        def add_function_e2e(md_, desc_, n_, nc_):
            """fresh arrays every call (as the reference's addFunction allocates its three vectors inside the timed call)"""
            nodes = np.empty(n_); cells = np.empty((nc_, 32), np.uint32); cmap = np.empty(nc_, np.uint32); tm = np.zeros(6)
            capi.check(capi.lib.dg_add_function_sdf(md_.handle, C.byref(desc_), 1.0, capi.ptr(nodes, capi.F64P), capi.ptr(cells, capi.U32P), capi.ptr(cmap, capi.U32P), capi.ptr(tm, capi.F64P)))
            return nodes, cells, cmap, tm
        if world == 1:
            for _ in range(2):
                add_function_e2e(md, desc, n_nodes, n_cells)
            n_e2e = max(3, args.steps // 2)
            ts, tms = [], []
            for _ in range(n_e2e):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = add_function_e2e(md, desc, n_nodes, n_cells)
                ts.append(time.perf_counter() - t0); tms.append(out[3])
                del out
            dt = float(np.mean(ts))
            tm = np.mean(np.array(tms), axis=0)
            e2e = {"value": n_nodes / dt, "unit": "nodes/s", "h2d_bytes_per_step": C.sizeof(capi.GridDesc),
                   "d2h_bytes_per_step": 8 * n_nodes, "ms_per_step": dt * 1e3, "best_ms": min(ts) * 1e3,
                   "host_bytes_written_per_step": 8 * n_nodes + 132 * n_cells,
                   "breakdown_ms": {"total_inside_call": float(tm[0]), "node_pipeline_done": float(tm[1]), "coefficient_array_prefaulted": float(tm[3]),
                                    "host_worker_threads": int(tm[4]), "allocation_and_return": dt * 1e3 - float(tm[0])},
                   "api": "dg_add_function_sdf(mesh, grid, sign, nodes_host, cells_host, cell_map_host): the whole of addFunction (:780-899) into fresh "
                          "pageable host arrays -- K1 chunks on two streams, D2H through a pooled pinned double buffer, connectivity table (:833-886) and "
                          "cell map (:888-891) written by host threads while the GPU works; the mesh/BVH was uploaded once by dg_mesh_create (as "
                          "TriangleMeshDistance is built once, outside addFunction's timer, in the reference)",
                   "mesh_upload": {"host_build_ms": mesh_info["build_us"] / 1e3, "h2d_ms": mesh_info["upload_us"] / 1e3, "h2d_bytes": mesh_info["device_bytes"]}}
        else:
            # one process per GPU: every rank delivers its node-id chunks to its own host buffers (dg_sample_sdf) ...
            my_ranges = [(b, e) for (_j, b, e) in my_chunks if e > b] if args.sharding != "slab" else [(b, e) for (b, e) in sdf_sampler.sh.ranges[rank] if e > b]
            outs = [np.empty(e - b) for (b, e) in my_ranges]

            def e2e_step():
                for (b, e), o in zip(my_ranges, outs):
                    capi.check(capi.lib.dg_sample_sdf(md.handle, C.byref(desc), 1.0, b, e, capi.ptr(o, capi.F64P)))
            for _ in range(2):
                e2e_step()
            barrier()
            t0 = time.perf_counter()
            n_e2e = max(3, args.steps // 2)
            for _ in range(n_e2e):
                e2e_step()
            torch.cuda.synchronize()
            dt = max_over_ranks((time.perf_counter() - t0) / n_e2e)
            e2e = {"value": n_nodes / dt, "unit": "nodes/s", "h2d_bytes_per_step": C.sizeof(capi.GridDesc) * len(my_ranges),
                   "d2h_bytes_per_step": 8 * n_nodes, "ms_per_step": dt * 1e3,
                   "api": "one process per GPU: dg_sample_sdf(mesh, grid, sign, l_begin, l_end, out_host) per rank over its node-id chunks (kernel + D2H into pageable host buffers)"}
            # ... and the single-process form a C++ caller uses: rank 0 drives ALL N GPUs through dg_add_function_sdf_multi while the other ranks idle
            barrier()
            dist.barrier(group=cpu_group)
            if rank == 0:
                try:
                    grp = C.c_void_p()
                    capi.check(capi.lib.dg_mesh_group_create(md.handle, world, None, C.byref(grp)))
                    ts = []
                    for it in range(2 + 3):
                        nodes = np.empty(n_nodes); cells = np.empty((n_cells, 32), np.uint32); cmap = np.empty(n_cells, np.uint32); tm = np.zeros(6)
                        t0 = time.perf_counter()
                        capi.check(capi.lib.dg_add_function_sdf_multi(grp, C.byref(desc), 1.0, capi.ptr(nodes, capi.F64P), capi.ptr(cells, capi.U32P), capi.ptr(cmap, capi.U32P), capi.ptr(tm, capi.F64P)))
                        if it >= 2:
                            ts.append(time.perf_counter() - t0)
                    same = bool(np.array_equal(nodes.view(np.uint64), full[:n_nodes].cpu().numpy().view(np.uint64)))
                    e2e["single_process_c_abi"] = {"api": f"dg_add_function_sdf_multi(group of {world} GPUs, ...): whole addFunction from ONE process, host arrays out (what GenerateSDF --gpus N calls)",
                                                   "ms_per_step": float(np.mean(ts)) * 1e3, "value": n_nodes / float(np.mean(ts)), "unit": "nodes/s",
                                                   "node_pipeline_ms": float(tm[1]), "equals_sharded_result": same}
                    capi.lib.dg_mesh_group_destroy(grp)
                except Exception as ex:                          # an auxiliary leg must not take the bench line down
                    e2e["single_process_c_abi"] = {"error": repr(ex)}
            dist.barrier(group=cpu_group)                        # the idle ranks wait here, on the host
            barrier()

    # ---------------------------------------------------------------- interpolate half of the metric (config 4)
    interp = None
    if not args.no_interp:
        ires = [args.interp_resolution] * 3 if args.interp_resolution else INTERP["resolution"]
        idesc = dg.grid_desc(mn, mx, ires)
        nn = C.c_uint64(); capi.check(capi.lib.dg_grid_num_nodes(idesc.resolution, C.byref(nn))); nn = nn.value
        coeffs = torch.empty(nn, dtype=torch.float64, device=dev)
        sp = C.c_void_p(stream.cuda_stream)
        t0 = time.perf_counter()
        capi.check(capi.lib.dg_sample_sdf_device(md.handle, C.byref(idesc), 1.0, 0, nn, C.c_void_p(coeffs.data_ptr()), sp))
        torch.cuda.synchronize()
        build_s = time.perf_counter() - t0
        fh = C.c_void_p()
        capi.check(capi.lib.dg_field_create_device(C.byref(idesc), C.c_void_p(coeffs.data_ptr()), nn, sp, C.byref(fh)))
        torch.cuda.synchronize()
        del coeffs
        nq = INTERP["queries"]
        q_lo = (nq * rank) // world; q_hi = (nq * (rank + 1)) // world
        xh = splitmix_points(nq, INTERP["seed"], mn, mx)[q_lo:q_hi]
        xh_t = torch.from_numpy(np.ascontiguousarray(xh)).pin_memory()
        xd = xh_t.to(dev)
        phi = torch.empty(q_hi - q_lo, dtype=torch.float64, device=dev)
        grad = torch.empty((q_hi - q_lo, 3), dtype=torch.float64, device=dev)

        def interp_step(with_grad=True):
            capi.check(capi.lib.dg_interpolate_batch_device(fh, C.c_void_p(xd.data_ptr()), q_hi - q_lo, C.c_void_p(phi.data_ptr()),
                                                            C.c_void_p(grad.data_ptr()) if with_grad else None, sp))
        ig_ms, _ = timed(lambda: interp_step(True), 20, 3)
        iv_ms, _ = timed(lambda: interp_step(False), 20, 3)
        ig_ms, iv_ms = float(np.mean(ig_ms)), float(np.mean(iv_ms))
        # SURVEY 8(d) config 4: the same points sorted by cell (z-major cell index) separate gather locality from arithmetic
        cell = ((xh - mn) / (mx - mn) * ires[0]).astype(np.int64).clip(0, ires[0] - 1)
        order = np.argsort((cell[:, 2] * ires[1] + cell[:, 1]) * ires[0] + cell[:, 0], kind="stable")
        xd_sorted = torch.from_numpy(np.ascontiguousarray(xh[order])).to(dev)
        xd_keep = xd
        xd = xd_sorted
        is_ms, _ = timed(lambda: interp_step(True), 20, 3)
        is_ms = float(np.mean(is_ms))
        xd = xd_keep
        del xd_sorted
        interp_step(True); torch.cuda.synchronize()          # phi / grad hold the unsorted queries' results again (compared with the host path below)
        if args.dump_outputs and rank == 0:
            qi = torch.from_numpy(dump_sample(q_hi - q_lo, DUMP["queries"], DUMP["seed"])).to(dev)
            dumped["interpolate_phi"] = phi[qi].cpu().numpy()
            dumped["interpolate_grad"] = grad[qi].cpu().numpy()
            del qi
        alg = 312.0 * (q_hi - q_lo)
        gbs = alg / (ig_ms * 1e-3) / 1e9
        # e2e through the host API: page-locked host buffers (the contract's pinned inputs), H2D + kernel + D2H inside the timed region
        ph_t = torch.empty(q_hi - q_lo, dtype=torch.float64).pin_memory(); gh_t = torch.empty((q_hi - q_lo, 3), dtype=torch.float64).pin_memory()
        xq, ph, gh = xh_t.numpy(), ph_t.numpy(), gh_t.numpy()

        def host_call(x_, p_, g_):
            capi.check(capi.lib.dg_interpolate_batch(fh, capi.ptr(x_, capi.F64P), len(x_), capi.ptr(p_, capi.F64P), capi.ptr(g_, capi.F64P)))
        for _ in range(2):
            host_call(xq, ph, gh)
        barrier(); t0 = time.perf_counter()
        for _ in range(5):
            host_call(xq, ph, gh)
        dt = max_over_ranks((time.perf_counter() - t0) / 5)
        pinned_equal = bool(np.array_equal(ph.view(np.uint64), phi.cpu().numpy().view(np.uint64)))
        # the same with ordinary (pageable) numpy arrays: staged through the library's pinned pool
        xp, pp, gp = np.array(xq), np.empty(len(xq)), np.empty((len(xq), 3))
        host_call(xp, pp, gp)
        barrier(); t0 = time.perf_counter()
        for _ in range(3):
            host_call(xp, pp, gp)
        dt_pageable = max_over_ranks((time.perf_counter() - t0) / 3)
        del xp, pp, gp
        interp = {"metric": "interpolate()+gradient Mqueries/s", "value": nq / (ig_ms * 1e-3) / 1e6, "unit": "Mqueries/s",
                  "value_only_mqps": nq / (iv_ms * 1e-3) / 1e6, "cell_sorted_mqps": nq / (is_ms * 1e-3) / 1e6, "ms_per_launch": ig_ms, "queries": nq,
                  "config": {"workload": f"10M splitmix64 uniform queries (seed 0x5EED) on the {ires[0]}^3 SDF of the headline mesh "
                                         f"({nn} nodes; packed cell blocks {16 * ires[0] * ires[1] * ires[2] * 16 / 1e9:.2f} GB >> L2)",
                             "field_build_s": build_s},
                  "roofline": {"kernel": "interpolate_kernel<true> (K2)", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm_gbs"],
                               "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": NCU["k2_dram_bytes_per_launch"], "traffic_source": NCU["k2_source"],
                               "peak_source": peak_src, "algorithmic_bytes_per_query": 312, "algorithmic_bytes_per_launch": alg},
                  "e2e": {"value": nq / dt / 1e6, "unit": "Mqueries/s", "h2d_bytes_per_step": 24 * nq, "d2h_bytes_per_step": 32 * nq, "ms_per_step": dt * 1e3,
                          "pcie_gbs": 56.0 * (q_hi - q_lo) / dt / 1e9, "equals_device_result": pinned_equal,
                          "pageable_buffers": {"value": nq / dt_pageable / 1e6, "unit": "Mqueries/s", "ms_per_step": dt_pageable * 1e3},
                          "api": "dg_interpolate_batch(field, x_host, n, phi_host, grad_host): 3-slot pipeline of 512k-query chunks (H2D, kernel, D2H overlapped); "
                                 "page-locked caller buffers are DMA'd directly, pageable ones are staged through pooled pinned buffers"}}
        del ph_t, gh_t
        capi.lib.dg_field_destroy(fh)
        del phi, grad, xd, xd_keep
        torch.cuda.empty_cache()
        if rank == 0 and world == 1 and not args.no_cpu:
            c = run_cpu_child({"what": "interp", "mesh": source, "torus": WORKLOAD["torus"], "res": ires, "queries": nq, "seed": INTERP["seed"], "runs": 2})
            if "seconds" in c:
                c["value"] = nq / c["seconds"] / 1e6; c["unit"] = "Mqueries/s"
            interp["cpu_baseline"] = c

    # ---------------------------------------------------------------- north-star target config: 256^3 grid, 100,000-triangle mesh
    target = None
    if not args.no_target:
        tmesh, ttext, _ = workload_mesh(dg, "target")
        tmd = dg.TriangleMeshDistance(tmesh)
        tmn, tmx = dg.generate_sdf_domain(tmesh.vertices)
        tres = [args.target_resolution] * 3
        tdesc = dg.grid_desc(tmn, tmx, tres)
        tn = C.c_uint64(); capi.check(capi.lib.dg_grid_num_nodes(tdesc.resolution, C.byref(tn))); tn = tn.value
        tsampler = make_sampler(tmd, tdesc, tn)
        tfull = torch.empty(tsampler.sh.padded, dtype=torch.float64, device=dev)
        t_ms, _ = timed(lambda: tsampler.step(tfull), 3, 1)
        t_ms = float(np.mean(t_ms))
        target = {"workload": f"north_star target: {tres[0]}^3 grid ({tn} nodes), {ttext}, strong scaling, sharding as config.parallelism",
                  "ms_per_step": t_ms, "value": tn / (t_ms * 1e-3), "unit": "nodes/s",
                  "n_gpus": world, "sharded_equals_single_launch": same_as_single_launch(tmd, tdesc, tn, tfull)}
        del tfull, tsampler
        torch.cuda.empty_cache()
        if world == 1 and not args.no_e2e:
            tnc = tres[0] ** 3
            add_function_e2e(tmd, tdesc, tn, tnc)
            ts, tms = [], []
            for _ in range(3):
                torch.cuda.synchronize(); t0 = time.perf_counter()
                out = add_function_e2e(tmd, tdesc, tn, tnc)
                ts.append(time.perf_counter() - t0); tms.append(out[3]); del out
            tm = np.mean(np.array(tms), axis=0)
            target["e2e"] = {"api": "dg_add_function_sdf: whole addFunction into fresh host arrays (as `e2e` above)", "ms_per_step": float(np.mean(ts)) * 1e3, "best_ms": min(ts) * 1e3,
                             "value": tn / float(np.mean(ts)), "unit": "nodes/s", "d2h_bytes_per_step": 8 * tn, "host_bytes_written_per_step": 8 * tn + 132 * tnc,
                             "breakdown_ms": {"total_inside_call": float(tm[0]), "node_pipeline_done": float(tm[1]), "coefficient_array_prefaulted": float(tm[3]),
                                              "host_worker_threads": int(tm[4]), "allocation_and_return": float(np.mean(ts)) * 1e3 - float(tm[0])}}
        if rank == 0 and world == 1 and not args.no_cpu:
            c = addfunction_baseline("target", None, tres, runs=1, warm=0, max_seconds=args.cpu_seconds, check_gpu=False, stats_nodes=2000)
            target["cpu_baseline"] = c
            if "value" in c and "e2e" in target:
                target["e2e_speedup_vs_cpu_baseline"] = target["e2e"]["value"] / c["value"]
        del tmd

    # ---------------------------------------------------------------- the reference's other meshes (configs 3/5), when staged
    real = None
    if not args.no_real and os.path.isdir(RES_DIR):
        real = []
        for name, r3 in (("dragon", 256), ("happy_buddha", 256)):
            path = os.path.join(RES_DIR, name + ".obj")
            if not os.path.exists(path):
                continue
            rmesh = dg.TriangleMesh(path)
            t0 = time.perf_counter(); rmd = dg.TriangleMeshDistance(rmesh); t_create = time.perf_counter() - t0
            rmn, rmx = dg.generate_sdf_domain(rmesh.vertices)
            r3 = args.real_resolution or r3
            rdesc = dg.grid_desc(rmn, rmx, [r3] * 3)
            rn = C.c_uint64(); capi.check(capi.lib.dg_grid_num_nodes(rdesc.resolution, C.byref(rn))); rn = rn.value
            rs = make_sampler(rmd, rdesc, rn)
            rfull = torch.empty(rs.sh.padded, dtype=torch.float64, device=dev)
            r_ms, _ = timed(lambda: rs.step(rfull), 2, 1)
            r_ms = float(np.mean(r_ms))
            entry = {"mesh": name + ".obj", "triangles": int(rmesh.nFaces()), "grid": r3, "nodes": rn, "ms_per_step": r_ms, "value": rn / (r_ms * 1e-3),
                     "unit": "nodes/s", "mesh_create_s": t_create, "watertight_flags": rmd.info()["watertight_flags"]}
            if rank == 0 and world == 1 and not args.no_cpu:
                # bounded CPU sample of the reference on the real mesh + a strided full-size parity check of the GPU array against it
                sys.path.insert(0, os.path.join(ROOT, "tests"))
                entry["cpu_baseline"] = addfunction_baseline(name, None, [r3] * 3, runs=1, warm=0, max_seconds=min(10.0, args.cpu_seconds), check_gpu=False, stats_nodes=0)
                entry["parity_strided"] = strided_parity(rmesh, rmn, rmx, [r3] * 3, rfull[:rn], 1_000_000)
            if name == "dragon" and world == 1 and not args.no_density:      # config 5: GenerateDensityMap on the dragon SDF, h = 0.1, rho0 = 1000
                fh = C.c_void_p(); sp = C.c_void_p(stream.cuda_stream)
                capi.check(capi.lib.dg_field_create_device(C.byref(rdesc), C.c_void_p(rfull.data_ptr()), rn, sp, C.byref(fh)))
                dens = torch.empty(rn, dtype=torch.float64, device=dev)
                k3_ms, _ = timed(lambda: capi.check(capi.lib.dg_density_map_device(fh, 0.1, 1000.0, 0, 0, rn, C.c_void_p(dens.data_ptr()), sp)), 1, 1)
                active = int(((dens > 0) & (dens < 1e300)).sum().item())
                entry["density_map"] = {"h": 0.1, "rho0": 1000.0, "ms": float(k3_ms[0]), "value": rn / (k3_ms[0] * 1e-3), "unit": "nodes/s",
                                        "nodes_in_quadrature_branch": active, "fp64_roofline": k3_roofline(active, float(k3_ms[0]), fp64_peak)}
                capi.lib.dg_field_destroy(fh); del dens
            real.append(entry)
            del rfull, rs, rmd
            torch.cuda.empty_cache()

    # ---------------------------------------------------------------- density map (config 5 kernel) on the headline SDF, N = 1 only
    density = None
    if world == 1 and not args.no_density:
        sdf_sampler.launch(full); torch.cuda.synchronize()
        fh = C.c_void_p()
        sp = C.c_void_p(stream.cuda_stream)
        capi.check(capi.lib.dg_field_create_device(C.byref(desc), C.c_void_p(full.data_ptr()), n_nodes, sp, C.byref(fh)))
        dens = torch.empty(n_nodes, dtype=torch.float64, device=dev)
        h_dm = 0.1 * float(np.max(mx - mn)) / 2.5            # the reference default h = 0.1 is for a ~2.5-unit dragon

        def dm_step():
            capi.check(capi.lib.dg_density_map_device(fh, h_dm, 1000.0, 0, 0, n_nodes, C.c_void_p(dens.data_ptr()), sp))
        dm_ms, _ = timed(dm_step, 2, 1)
        dm_ms = float(np.mean(dm_ms))
        dens_h = dens.cpu().numpy()
        active = int(((dens_h > 0) & (dens_h < 1e300)).sum())
        density = {"metric": "GenerateDensityMap nodes/s (K3)", "value": n_nodes / (dm_ms * 1e-3), "unit": "nodes/s", "ms": dm_ms,
                   "config": {"workload": f"density_func + predicate over the {res[0]}^3 SDF above, h = {h_dm:.4f}, rho0 = 1000, 16^3 Gauss points",
                              "nodes_in_quadrature_branch": active},
                   "fp64_roofline": k3_roofline(active, dm_ms, fp64_peak)}
        if not args.no_cpu:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            from oracle_api import Oracle
            orc = Oracle()
            gd, r = orc.grid_desc(mn, mx, res)
            coeff_h = full[:n_nodes].cpu().numpy()
            t_cpu, n_cpu, ok = 0.0, 0, True
            for k in range(8):                                 # eight 192-node windows spread over the node index space
                l0 = int((k + 0.5) * n_nodes / 8); l1 = min(l0 + 192, n_nodes)
                t0 = time.perf_counter()
                ref = orc.density_map(gd, r, coeff_h, h_dm, 1000.0, False, l0, l1)
                t_cpu += time.perf_counter() - t0; n_cpu += l1 - l0
                ok = ok and np.array_equal(ref.view(np.uint64), dens_h[l0:l1].view(np.uint64))
            density["cpu_baseline"] = {"value": n_cpu / t_cpu, "unit": "nodes/s", "kind": "port", "cores": orc.max_threads(),
                                       "sample": f"{n_cpu} nodes in 8 windows, oracle/dg_oracle.cpp (the reference tool needs Eigen)",
                                       "bit_exact_vs_gpu": bool(ok)}
        try:                                                    # N3: the step after the density map in GenerateDensityMap
            cells_h = np.empty((n_cells, 32), np.uint32)
            capi.check(capi.lib.dg_build_cells(desc.resolution, 0, len(cells_h), capi.ptr(cells_h, capi.U32P)))
            density["reduce_field"] = reduce_field_leg(capi, desc, dens_h, cells_h, 0.0, 3000.0, with_reference=not args.no_cpu)
            del cells_h
        except Exception as ex:                                 # an auxiliary leg must not take the bench line down
            density["reduce_field"] = {"error": repr(ex)}
        capi.lib.dg_field_destroy(fh)
        del dens

    if world > 1 and not args.no_density:                      # N > 1: the same node function over node-id chunks + the SDF's all-gather
        from discregrid_b200.distributed import ShardedDensityMap
        sdf_sampler.step(full); torch.cuda.synchronize()
        fh, dens, dmap, setup_err = C.c_void_p(), None, None, None
        sp = C.c_void_p(stream.cuda_stream)
        try:                                                    # anything that can fail on ONE rank only happens before the collective part
            capi.check(capi.lib.dg_field_create_device(C.byref(desc), C.c_void_p(full.data_ptr()), n_nodes, sp, C.byref(fh)))
            dmap = ShardedDensityMap(fh, n_nodes, rank, world)
            dens = torch.empty(dmap.sh.padded, dtype=torch.float64, device=dev)
            torch.cuda.synchronize()
        except Exception as ex:
            setup_err = repr(ex)
        if max_over_ranks(0.0 if setup_err is None else 1.0) == 0.0:
            h_dm = 0.1 * float(np.max(mx - mn)) / 2.5
            dm_ms, _ = timed(lambda: dmap.step(dens, h_dm, 1000.0), 2, 1)
            dm_ms = float(np.mean(dm_ms))
            density = {"metric": "GenerateDensityMap nodes/s (K3)", "value": n_nodes / (dm_ms * 1e-3), "unit": "nodes/s", "ms": dm_ms, "n_gpus": world,
                       "config": {"workload": f"density_func + predicate over the {res[0]}^3 SDF above, h = {h_dm:.4f}, rho0 = 1000, 16^3 Gauss points; "
                                              f"8 round-robin node-id chunks per rank + one in-place all-gather per row"}}
        else:
            density = {"error": setup_err or "setup failed on another rank"}
        if fh:
            capi.lib.dg_field_destroy(fh)
        del dens

    # ---------------------------------------------------------------- the rebuilt C++ tools as a user runs them (facade over the C-ABI), N = 1 only
    tools = None
    gen_sdf, gen_dm = os.path.join(ROOT, "build", "bin", "GenerateSDF"), os.path.join(ROOT, "build", "bin", "GenerateDensityMap")
    mesh_path = os.path.join(RES_DIR, "bunny.obj")
    if rank == 0 and world == 1 and not args.no_density and not args.no_e2e and os.path.exists(gen_sdf) and os.path.exists(gen_dm) and os.path.exists(mesh_path) and source == "bunny":
        try:
            tdir = scratch_dir()
            cdf, cdm = os.path.join(tdir, f"_dg_tools_{os.getpid()}.cdf"), os.path.join(tdir, f"_dg_tools_{os.getpid()}.cdm")
            rstr = f"{res[0]} {res[1]} {res[2]}"
            t0 = time.perf_counter(); r1 = subprocess.run([gen_sdf, "-r", rstr, "-o", cdf, mesh_path], capture_output=True, text=True, timeout=900); t_sdf = time.perf_counter() - t0
            h_tool = 0.1 * float(np.max(mx - mn)) / 2.5
            t0 = time.perf_counter(); r2 = subprocess.run([gen_dm, "-s", repr(h_tool), "-o", cdm, cdf], capture_output=True, text=True, timeout=1800); t_dm = time.perf_counter() - t0
            tools = {"what": "wall clock of the rebuilt reference tools, process start to exit (OBJ parse, BVH build + upload, CUDA context, addFunction, "
                             "K3 + both reduceField passes, file I/O): GenerateSDF -r 128^3 bunny.obj; GenerateDensityMap (with reduction) on its output",
                     "generate_sdf_s": t_sdf, "generate_sdf_rc": r1.returncode, "generate_density_map_s": t_dm, "generate_density_map_rc": r2.returncode,
                     "cdf_bytes": os.path.getsize(cdf) if os.path.exists(cdf) else None, "cdm_bytes": os.path.getsize(cdm) if os.path.exists(cdm) else None}
            for f_ in (cdf, cdm):
                if os.path.exists(f_):
                    os.remove(f_)
        except Exception as ex:
            tools = {"error": repr(ex)}

    # ---------------------------------------------------------------- CPU baseline (the reference's real addFunction), rank 0, N = 1 only
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu = addfunction_baseline(source, WORKLOAD["torus"], res, runs=2, warm=1, max_seconds=args.cpu_seconds, check_gpu=True)
        if "error" in cpu:
            cpu = {"value": None, "unit": "nodes/s", "cores": 0, "kind": "reference", "sample": "unavailable: " + cpu["error"][:200]}

    # ---------------------------------------------------------------- roofline of the dominant kernel (K1): fp64 issue, not HBM
    flops_node = (cpu or {}).get("flops_per_node") or NCU["k1_flops_per_node_fallback"]
    k1_flops = flops_node * my_nodes
    k1_tflops = k1_flops / (k1_ms * 1e-3) / 1e12
    k1_alg_bytes = 8.0 * my_nodes + mesh_info["device_bytes"]          # 8 B/node written + mesh records read once
    k1_gbs = k1_alg_bytes / (k1_ms * 1e-3) / 1e9
    roofline = {"kernel": "sdf_sample_nodes_kernel (K1)", "bound": "fp64", "achieved": k1_tflops, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": k1_tflops / fp64_peak if fp64_peak else None,
                "traffic": NCU["k1_dram_bytes_per_launch"] if (world == 1 and source == NCU["k1_mesh"] and res[0] == 128) else None, "traffic_source": NCU["k1_source"],
                "peak_source": "measured in this run: dg_fp64_rate_probe (8 independent DMUL+DADD chains per thread, 8 blocks of 256 threads per SM) -- "
                               "the library is built without FMA contraction (bit-exact parity with the reference's x86-64 build), so this, not the "
                               "FMA rate, is the ceiling of its fp64 pipe",
                "algorithmic_flops_per_node": flops_node,
                "algorithmic_flops_note": "SURVEY 8(d): visits * 24 + leaf tests * 65 of the REFERENCE algorithm (spheres only, all in fp64), counted by the "
                                          "oracle port on a strided node sample of this workload; the kernel itself does fewer (fp32 sphere filter, box skip)",
                "launches_per_step": n_launch, "avg_launch_ms": k1_ms / max(1, n_launch),
                "ncu": NCU["k1_summary"],
                "hbm": {"bound": "hbm", "achieved": k1_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": k1_gbs / peaks["hbm_gbs"], "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": k1_alg_bytes / max(1, n_launch),
                        "note": "K1 is not HBM-bound: BVH + triangle records are L2-resident, compulsory HBM traffic is 8 B/node (SURVEY 8d)"},
                "interpolate": (interp or {}).get("roofline")}
    if e2e is not None and interp is not None:
        e2e["interpolate"] = interp["e2e"]
    if cpu is not None and interp is not None and "cpu_baseline" in interp:
        cpu["interpolate"] = interp["cpu_baseline"]

    if rank == 0:
        line = {"metric": "SDF grid nodes/sec (addFunction)", "value": value, "unit": "nodes/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": data, "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline, "cpu_baseline": cpu, "interpolate": interp, "target_config": target, "reference_meshes": real, "density_map": density, "tools_e2e": tools,
                "timing": {"per_step_ms": sdf_ms, "wall_s_timed_region": sdf_wall, "k1_only_ms_per_step": k1_ms,
                           "collective_and_unpack_ms": ms_step - k1_ms},
                "parity_full": None if cpu is None else {"nodes_bit_exact": cpu.get("parity_nodes_bit_exact"), "nodes_compared": cpu.get("parity_nodes_compared"),
                                                         "cells_equal": cpu.get("parity_cells_equal"),
                                                         "interpolate_bit_exact": ((interp or {}).get("cpu_baseline") or {}).get("bit_exact_vs_gpu"),
                                                         "interpolate_queries_compared": ((interp or {}).get("cpu_baseline") or {}).get("queries_compared")},
                "sharded_equals_single_launch": sharded_ok,
                "library": {"path": os.path.relpath(capi.LIB_PATH, ROOT), "emulated": hasattr(capi.lib, "emu_mesh_create")}}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ncu-derived constants of the shipped kernels AT THE BENCH CONFIGURATIONS (profiles/: `ncu --set full --clock-control none`; numbers taken
# under ncu are never bench values -- these are per-launch DRAM bytes and pipe statistics only)
NCU = {
    "k1_mesh": "bunny", "k1_dram_bytes_per_launch": 48.75e6 + 83.26e6,
    "k1_source": "profiles/r2w_ncu_summary.csv: ncu --set full of the shipped sdf_sample_nodes_kernel (packet walk) at this configuration (bunny.obj, 128^3): dram read 48.8 MB "
                 "(mesh records) + write 83.3 MB (8 B/node; the rest of the 119 MB drains after the launch)",
    "k1_summary": {"capture": "profiles/r2w_ncu_summary.csv (bunny.obj 128^3, 34.1 ms under ncu; the per-lane kernel of round 1: r2a, 76.9 ms)",
                   "warp_instructions": 29.5e9, "warp_instructions_per_lane_kernel": 60.4e9, "lanes_active_per_instruction": 28.6, "issue_active_pct": 74.9,
                   "fp64_pipe_pct": 7.2, "alu_pipe_pct": 44.1, "warps_active_pct": 37.6, "registers": 72, "shared_kb_per_block": 15.0, "l1_hit_pct": 56.2, "l2_hit_pct": 94.4,
                   "instruction_shares": "(r2v capture, same walk) node step 43 %, certified fp32 triangle bound 23 %, exact fp64 triangle test 7.5 %, deferred-child re-test 7 %, "
                                         "candidate list 6 %, index arithmetic + sign 8 %, reference-order replay 3 %, per-lane fallback 0.1 %",
                   "reading": "instruction-issue bound (75 % of the issue slots busy, 28.6 of 32 lanes) with half the instructions of the per-lane kernel; neither HBM (0.03 %), "
                              "the fp64 pipe (7 %) nor the L1 data pipe (41 %)"},
    "k1_flops_per_node_fallback": 15800.0,
    "k2_dram_bytes_per_launch": 2757.4e6 + 312.9e6,
    "k2_source": "profiles/r2a_ncu_summary.csv: ncu --set full of interpolate_kernel<true>, 10 M queries on the 256^3 field: dram read 2.757 GB + write 0.313 GB = 3.07 GB "
                 "against 3.12 GB algorithmic (no re-reads); fp64 pipe 59 %, 32 of 32 lanes",
}


def k3_roofline(active_nodes, ms, fp64_peak):
    """K3 against the measured fp64 issue rate.  Work counted per node in the quadrature branch: one value-only interpolation (~155 unfused
    flops, SURVEY 8d) + the kernel/gamma arithmetic (~15) for every Gauss point INSIDE the kernel support |xi| <= h -- the points outside
    contribute exactly +0 and the kernel skips them (the reference evaluates all 4096)."""
    x, _w = np.polynomial.legendre.leggauss(16)
    inside = int((x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2 <= 1.0).sum())
    flops = float(inside) * (155.0 + 15.0) * active_nodes
    t = flops / (ms * 1e-3) / 1e12
    return {"bound": "fp64", "achieved": t, "peak": fp64_peak, "unit": "TFLOP/s", "frac": t / fp64_peak if fp64_peak else None,
            "algorithmic_flops_per_active_node": inside * 170, "gauss_points_inside_support": inside, "gauss_points": 4096,
            "peak_source": "dg_fp64_rate_probe (DMUL+DADD, no FMA), this run",
            "ncu": "profiles/r2a_ncu_summary.csv (128^3 bunny field, before K3_FAST_DIV): fp64 pipe 29.5 %, issue active 26.6 %, 26.8 of 32 lanes, long-scoreboard bound"}


def strided_parity(mesh, mn, mx, res, d_nodes, n_check):
    """full-size parity sample: `n_check` evenly strided nodes of a device-resident coefficient array vs the reference's own
    signed_distance (oracle/_ref/libdgref.so, else the oracle port) at the oracle's node positions -- bit for bit"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_api import Oracle, RefMesh, have_ref
    import torch
    orc = Oracle()
    gd, r = orc.grid_desc(mn, mx, res)
    n = orc.num_nodes(r)
    ids = np.unique(np.linspace(0, n - 1, min(n, n_check)).astype(np.int64))
    x = orc.node_positions_at(gd, r, ids)
    m = RefMesh(mesh.vertices, mesh.faces) if have_ref() else orc.mesh(mesh.vertices, mesh.faces)
    want = m.sample_points(x) if have_ref() else m.distance(x)[0]
    got = d_nodes[torch.from_numpy(ids).to(d_nodes.device)].cpu().numpy()
    return {"nodes_compared": int(len(ids)), "bit_exact": bool(np.array_equal(got.view(np.uint64), want.view(np.uint64))),
            "against": "reference TriangleMeshDistance.h (oracle/_ref)" if have_ref() else "oracle port"}


def reduce_field_leg(capi, desc, values, cells, lo, hi, with_reference, tmp_dir=None):
    """SURVEY 8(f) N3: reduceField(field, lo <= v <= hi) (cmd/generate_density_map/main.cpp:141-144) on a sampled field:
    dg_reduce_field vs the reference class's own reduceField (oracle/_ref, when built)."""
    if tmp_dir is None:
        tmp_dir = scratch_dir()
    keep = np.ascontiguousarray((lo <= values) & (values <= hi) & (values != np.finfo(np.float64).max), np.uint8)
    n_grid_cells = int(desc.resolution[0]) * int(desc.resolution[1]) * int(desc.resolution[2])
    best, out = None, None
    for _ in range(3):
        nodes, cc = values.copy(), cells.copy()
        cmap = np.empty(n_grid_cells, np.uint32); n1, n2 = C.c_uint64(), C.c_uint64(); tm = np.zeros(5)
        t0 = time.perf_counter()
        capi.check(capi.lib.dg_reduce_field(C.byref(desc), capi.ptr(nodes, capi.F64P), len(nodes), keep.ctypes.data_as(C.POINTER(C.c_uint8)),
                                            capi.ptr(cc, capi.U32P), len(cc), capi.ptr(cmap, capi.U32P), 0, C.byref(n1), C.byref(n2), capi.ptr(tm, capi.F64P)))
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, out = dt, (nodes[:n1.value], cc[:n2.value], cmap, tm.copy())
    leg = {"what": "reduceField of the density field with the tool's predicate 0 <= v <= 3 rho0 (dg_reduce_field)",
           "nodes_in": int(len(values)), "nodes_out": int(len(out[0])), "cells_in": int(len(cells)), "cells_out": int(len(out[1])),
           "ms": best * 1e3, "ms_cells_nodes_sort_write": [float(t) for t in out[3][:4]], "morton_keys_tied": bool(out[3][4])}
    if with_reference:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from oracle_api import REF_GRID_SO, RefGrid
        if os.path.exists(REF_GRID_SO):
            import struct
            src, dst = os.path.join(tmp_dir, f"dg_reduce_in_{os.getpid()}.cdf"), os.path.join(tmp_dir, f"dg_reduce_out_{os.getpid()}.cdf")
            try:
                with open(src, "wb") as f:                              # the reference's one-field file layout (:678-719)
                    f.write(struct.pack("<3d", *desc.domain_min)); f.write(struct.pack("<3d", *desc.domain_max)); f.write(struct.pack("<3I", *desc.resolution))
                    f.write(struct.pack("<3d", *desc.cell_size)); f.write(struct.pack("<3d", *desc.inv_cell_size)); f.write(struct.pack("<QQ", n_grid_cells, 1))
                    for arr in (values, cells, np.arange(len(cells), dtype=np.uint32)):
                        f.write(struct.pack("<QQ", 1, len(arr))); f.write(np.ascontiguousarray(arr).tobytes())
                ref = RefGrid(src); t_ref = ref.reduce_window(0, lo, hi); ref.save(dst); ref.close()
                raw = np.fromfile(dst, np.uint8)
                off = 24 * 4 + 12 + 16                                   # header: 4 x 3 doubles, 3 uint32, n_cells, n_fields

                def nested(dtype, width):
                    nonlocal off
                    n = int(raw[off + 8:off + 16].view(np.uint64)[0]); off += 16
                    a = raw[off:off + n * width * np.dtype(dtype).itemsize].view(dtype); off += a.nbytes
                    return a.reshape(n, width) if width > 1 else a
                rn, rc, rm = nested(np.float64, 1), nested(np.uint32, 32), nested(np.uint32, 1)
                same = bool(np.array_equal(rn.view(np.uint64), out[0].view(np.uint64)) and np.array_equal(rc, out[1]) and np.array_equal(rm, out[2]))
                leg["reference"] = {"ms": t_ref * 1e3, "kind": "reference", "impl": "CubicLagrangeDiscreteGrid::reduceField of oracle/_ref (serial, one std::set per node)",
                                    "identical_nodes_cells_cell_map": same, "speedup": t_ref / best}
            finally:
                for p_ in (src, dst):
                    if os.path.exists(p_):
                        os.remove(p_)
    return leg


if __name__ == "__main__":
    main()
