"""The library's CUDA kernels on a machine without a GPU: edyn_b200/csrc compiled against tests/emu (a CPU emulation of
blocks, __syncthreads, warp collectives, cooperative launches and the ticket polls -- see tests/emu/include/cuda_runtime.h
for what it is and is not) and driven through the real C ABI and Python adapter, in lock step with the oracle.

It complements the -m gpu suite, it does not replace it: it executes the same C++ on the same data layout, so logic
errors show up; memory ordering, occupancy and speed do not exist here.  What it adds is CONTENT the GPU suite has not
seen: arbitrarily oriented static boxes, static / kinematic spheres and capsules, rotating kinematic bodies, hinges with
non-parallel axes and pivots that start apart, tilted ground planes, restitution up to 1, friction 0-2, 1-20 velocity and
0-6 position iterations -- through both solver schedules (island tiles and ticket dataflow)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(kind, first, last, tiles="1", steps=80, restitution=False, mutate=False):
    cmd = [sys.executable, os.path.join(ROOT, "tests", "emu", "lockstep.py"), kind, str(first), str(last), "--tiles", tiles, "--steps", str(steps)]
    if restitution:
        cmd.append("--restitution")
    if mutate:
        cmd.append("--mutate")
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=1500)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])["results"]


def test_emulation_primitives(tmp_path):
    """The emulation itself: barriers, warp collectives with full / partial masks and exited lanes, atomics, shared memory,
    the cub stand-ins, warps of one block waiting for each other through polled flags (tests/emu/selftest.cpp)."""
    import shutil
    cxx = shutil.which("g++")
    assert cxx
    exe = str(tmp_path / "emu_selftest")
    emu = os.path.join(ROOT, "tests", "emu")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I" + os.path.join(emu, "include"), "-o", exe, os.path.join(emu, "selftest.cpp"),
                    os.path.join(emu, "emu_runtime.cpp")], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "emu selftest ok" in out.stdout, out.stdout + out.stderr


def test_emulated_kernels_on_the_benchmark_scene_families(O):
    """Validates the emulation itself: these five are green on a real B200 (tests/test_gpu_parity.py)."""
    for res in _run("fixed", 0, 5, steps=60):
        assert res["ok"] and res["worst"] <= 1e-5, res
    assert sum(r["points"] for r in _run("fixed", 1, 2, steps=60)) > 50


@pytest.mark.parametrize("kind,first,last,tiles", [("narrow", 0, 2, "1"), ("wide", 0, 4, "1"), ("wide", 4, 6, "0"), ("narrow", 2, 3, "0")])
def test_emulated_kernels_on_random_scenes(O, kind, first, last, tiles):
    for res in _run(kind, first, last, tiles=tiles):
        assert res["ok"] and res["worst"] <= 1e-5, res


def test_emulated_restitution_solver(O):
    """B2D_FLAG_RESTITUTION_SOLVER (k_rest_* in b2d_kernels.cuh: the entity graph as adjacency lists, one thread per island
    walking it breadth first) against the oracle's restatement of restitution_solver.cpp -- which is bit-identical to the
    real stepper (tests/test_ref_stepper.py).  The device fixes the orders the reference inherits from EnTT (neighbours in
    ascending body id, ties of the fastest manifold to the smaller pair key); the oracle's defaults are those conventions."""
    for res in _run("fixed", 3, 4, restitution=True) + _run("narrow", 0, 2, restitution=True) + _run("wide", 0, 3, restitution=True):
        assert res["ok"] and res["worst"] <= 1e-5, res


def test_emulated_kernels_under_user_interference(O):
    """b2d_remove_bodies, b2d_add_bodies, b2d_remove_exclusions and b2d_upload_bodies every 13th step of random scenes."""
    for res in _run("narrow", 0, 2, steps=100, mutate=True):
        assert res["ok"] and res["points"] >= 6, res


def test_emulated_kernels_against_the_real_stepper_directly(O):
    """Kernels (emulated) vs the reference's real stepper_sequential (states recorded in tests/golden/ref_runs.npz), both
    free-running, nothing replayed: the hinge-chain family (config 5) within 1e-6 after 300 steps (measured 5e-10;
    north_star asks for 1e-4 relative after 1000), hello_world identical during the fall."""
    for res in _run("vsref", 0, 0):
        if res["scene"] == "hello_world":
            assert res["dpos"] == 0.0 and res["dvel"] == 0.0, res
        else:
            assert res["dpos"] <= 1e-6 and res["dvel"] <= 1e-6, res
