"""Rehearsal of the `-m gpu` suite on the CPU.  build/bin/libdgemu.so is the whole product library with every kernel run by tests/emu
(lanes as fibers) and the CUDA runtime stubbed on host memory.  With DISCREGRID_B200_LIB pointing at it -- and LD_PRELOAD, so that the
rebuilt C++ tools resolve the C-ABI there too -- the GPU tests that need neither torch nor a full-size grid run unchanged: kernels,
launchers, C-ABI layer, Python mirror, C++ facade and tools against the same goldens as on the B200.  A failure here means the GPU
run at the end of the round would fail for a reason that has nothing to do with the GPU.  (Not a CPU fallback: test infrastructure.)"""
import os
import subprocess
import sys

import pytest

from conftest import ROOT

EMU = os.path.join(ROOT, "build", "bin", "libdgemu.so")
FILES = ["tests/test_gpu_k1_sdf.py", "tests/test_gpu_k2_interp.py", "tests/test_gpu_k3_density.py", "tests/test_gpu_reference_tools.py",
         "tests/test_gpu_cpp_facade.py", "tests/test_gpu_multi_capi.py", "tests/test_gpu_reduce_field.py"]
# left to the real GPU: device tensors through torch, the full-size configuration, the 69k-855k-triangle meshes (minutes when emulated)
SKIP = "not large_grid and not host_pipeline and not device_form and not full_size and not slab_parts and not interleaved_parts and not reference_meshes_vs_oracle"


def test_gpu_suite_passes_on_the_emulated_library():
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    # DG_HOST_HELPERS_MIN_BYTES: dg_sample_sdf hands ranges of >= 32 MiB to pre-fault / copy workers; lowered so that the toy ranges take that path too
    env = dict(os.environ, DISCREGRID_B200_LIB=EMU, LD_PRELOAD=EMU, DG_ALLOW_EMULATED_LIBRARY="1", DG_HOST_HELPERS_MIN_BYTES="4096")
    r = subprocess.run([sys.executable, "-m", "pytest", "-m", "gpu", "-q", "-x", "-k", SKIP, "-p", "no:cacheprovider"] + FILES,
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)
    tail = (r.stdout + r.stderr)[-3000:]
    assert r.returncode == 0, tail
    assert " passed" in r.stdout and "failed" not in r.stdout, tail


def test_multi_gpu_worker_on_two_gloo_ranks(tmp_path):
    """the worker script of tests/test_gpu_multi.py (node-id chunks, slabs, interleaved plane pairs, sharded density map, each compared
    with a single launch) on two gloo ranks with host tensors against the emulated library: the N > 1 plumbing end to end"""
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    from test_gpu_multi import WORKER
    script = tmp_path / "w.py"
    script.write_text(f"ROOT = {ROOT!r}\n" + WORKER)
    env = dict(os.environ, DISCREGRID_B200_LIB=EMU, DG_ALLOW_EMULATED_LIBRARY="1", DG_REHEARSAL="1", MASTER_ADDR="127.0.0.1", MASTER_PORT="29641")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29641", str(script)], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0 and "MULTI_OK 2" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]


def _bench_line(stdout):
    import json
    lines = [l for l in stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, stdout[-2000:]
    return json.loads(lines[0])


TOY = ["--steps", "2", "--warmup", "3", "--resolution", "6", "--interp-resolution", "5", "--target-resolution", "4", "--real-resolution", "3",
       "--cpu-seconds", "0.2"]


def test_smoke_entry_point_on_the_emulated_library():
    """__graft_entry__.smoke() (K1 + K2 + K3 against the oracle through the C-ABI) as the driver will call it, kernels emulated"""
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    r = subprocess.run([sys.executable, "-c", "import __graft_entry__ as g; g.smoke()"], cwd=ROOT, env=dict(os.environ, DISCREGRID_B200_LIB=EMU, DG_ALLOW_EMULATED_LIBRARY="1"),
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "smoke OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_bench_runs_end_to_end_single_rank(tmp_path):
    """bench.py, every leg, at toy sizes (tests/emu/bench_rehearsal.py: torch's CUDA surface on host stand-ins, emulated kernels): one JSON
    line with the contract's keys; the legs that self-check (interpolate / density vs the CPU references, reduceField vs the reference
    class) report agreement.  The reference-mesh leg runs on a small stand-in (tests/golden/sphere.obj staged as dragon.obj), and
    --dump-outputs writes the sampled outputs of the timed steps"""
    import shutil
    import numpy as np
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    meshes, out = tmp_path / "meshes", tmp_path / "out"
    meshes.mkdir()
    shutil.copy(os.path.join(ROOT, "tests", "golden", "sphere.obj"), meshes / "dragon.obj")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "emu", "bench_rehearsal.py")] + TOY + ["--dump-outputs", str(out)], cwd=ROOT,
                       env=dict(os.environ, DISCREGRID_B200_LIB=EMU, DG_ALLOW_EMULATED_LIBRARY="1", DG_BENCH_MESH_DIR=str(meshes)),
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    d = _bench_line(r.stdout)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["gpu_launches"] > 0 and d["value"] > 0 and d["e2e"]["value"] > 0
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"]) and {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert d["interpolate"]["cpu_baseline"]["bit_exact_vs_gpu"] is True
    assert d["target_config"]["value"] > 0 and len(d["reference_meshes"]) >= 1
    dumped = {p.name: np.load(p) for p in out.iterdir()}
    assert set(dumped) == {"sdf_nodes.npy", "interpolate_phi.npy", "interpolate_grad.npy"}
    assert all(a.dtype == np.float64 and np.isfinite(a).all() for a in dumped.values())
    assert len(dumped["sdf_nodes.npy"]) == d["config"]["nodes"] and dumped["interpolate_grad.npy"].shape == (len(dumped["interpolate_phi.npy"]), 3)
    red = d["density_map"]["reduce_field"]
    assert "error" not in red and red["nodes_out"] > 0
    if "reference" in red:
        assert red["reference"]["identical_nodes_cells_cell_map"] is True


@pytest.mark.parametrize("sharding", ["chunks", "interleaved"])
def test_bench_runs_end_to_end_two_ranks(sharding):
    """the same under torchrun with two gloo ranks: the N > 1 legs (sharded SDF + exchange, replicated interpolate, sharded density map)
    run, and the sharded coefficient arrays equal a single launch"""
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    port = {"chunks": "29661", "interleaved": "29663"}[sharding]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1", "--master-port", port,
                        os.path.join(ROOT, "tests", "emu", "bench_rehearsal.py"), "--gpus", "2", "--sharding", sharding, "--no-real"] + TOY, cwd=ROOT,
                       env=dict(os.environ, DISCREGRID_B200_LIB=EMU, DG_ALLOW_EMULATED_LIBRARY="1", MASTER_ADDR="127.0.0.1", MASTER_PORT=port), capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    d = _bench_line(r.stdout)
    assert d["n_gpus"] == 2 and d["sharded_equals_single_launch"] is True and d["target_config"]["sharded_equals_single_launch"] is True
    assert d["density_map"].get("ms", 0) > 0 and d["interpolate"]["value"] > 0


def test_package_refuses_the_emulated_library_by_default():
    """no accidental CPU path: pointing DISCREGRID_B200_LIB at the emulated test build without the rehearsal's explicit opt-in fails at import"""
    if not os.path.exists(EMU):
        pytest.skip("build/bin/libdgemu.so not built (make cpp)")
    env = {k: v for k, v in os.environ.items() if k != "DG_ALLOW_EMULATED_LIBRARY"}
    r = subprocess.run([sys.executable, "-c", "import discregrid_b200"], cwd=ROOT, env=dict(env, DISCREGRID_B200_LIB=EMU), capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "CPU-emulated TEST build" in r.stderr
