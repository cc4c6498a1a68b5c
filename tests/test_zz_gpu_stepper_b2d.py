"""The reference-side binding on the device: a REAL Edyn registry (edyn::attach, make_rigidbody,
make_constraint<hinge_constraint>, exclude_collision) stepped by edyn::stepper_b2d
(edyn_b200/csrc/host/stepper_b2d.hpp) over edyn_b200/libb2d.so must give exactly what the same scene gives when its
arrays are handed to the C ABI directly (edyn_b200.World) -- same library, same capacities, so bit for bit -- and must
follow the reference's own CPU stepper on the same user code.  tests/integration/_build/libedyn_b2d_dev.so is built where
the reference is (tests/integration/Makefile) and shipped; the CPU suite exercises the same harness over a mock
(tests/test_stepper_b2d.py).  Named to run after the parity suites."""
import numpy as np
import pytest

from tests.golden import make_ref_runs as R
from tests.golden import make_whole_step as G
from tests.test_stepper_b2d import EdynB2dWorld, _contacts_by_pair, build_integration, load

pytestmark = pytest.mark.gpu
MAX_MANIFOLDS = 1 << 16


@pytest.fixture(scope="module")
def dev(gpu, O):
    build_integration()
    lib = load(O, "dev")
    if lib is None:
        pytest.skip("tests/integration/_build/libedyn_b2d_dev.so not shipped (needs the reference at build time)")
    return lib


@pytest.mark.parametrize("name", ["boxes_27", "mixed_125", "chains_16"])
def test_registry_through_the_binding_equals_arrays_through_the_abi_on_device(dev, E, O, name):
    scene = G.build_scene(E, name)
    n = len(scene["bodies"]["kind"])
    nh = len(scene["hinges"]["a"]) if scene["hinges"] else 0
    w = EdynB2dWorld(O, dev, scene, max_manifolds=MAX_MANIFOLDS)
    d = E.scenes.build_world(scene, max_manifolds=MAX_MANIFOLDS, max_bodies=n + 8, max_hinges=max(nh, 1))
    for s in range(60):
        w.step(1); d.step(1)
        if s % 10 == 9:
            a, b = w.state(), d.download_state(aabb=True)
            for k in ("pos", "orn", "linvel", "angvel"):
                assert np.array_equal(a[k], b[k][:n]), f"{name} step {s}: {k} differs by {np.abs(a[k] - b[k][:n]).max():.3e}"
            moving = np.asarray(scene["bodies"]["kind"]) != 2        # static bodies keep the AABB make_rigidbody gave them
            assert np.array_equal(a["aabb"][moving], b["aabb"][:n][moving]), f"{name} step {s}: AABBs differ"
    assert d.stats()["error_flags"] == 0
    w.close(); d.close()


def test_device_contacts_mirrored_into_the_registry(dev, E, O):
    """stepper_b2d::mirror_contacts on the device: the registry's contact_manifold / contact_point entities, walked like
    user code walks them, hold exactly the device's manifolds (twin world fed the arrays directly)."""
    scene = G.build_scene(E, "mixed_125")
    n = len(scene["bodies"]["kind"])
    w = EdynB2dWorld(O, dev, scene, max_manifolds=MAX_MANIFOLDS)
    d = E.scenes.build_world(scene, max_manifolds=MAX_MANIFOLDS, max_bodies=n + 8, max_hinges=1)
    seen = 0
    for steps in (45, 5):
        w.step(steps); d.step(steps)
        (manifolds, points, created, destroyed), (started, ended) = w.mirror_contacts()
        got, want = w.r.contacts(), d.contacts()
        assert manifolds == len(want["pairs"]) and points == int(want["num"].sum()) and points > 100
        g = _contacts_by_pair(got, list(range(13)))
        t = _contacts_by_pair(want, [0, 1, 2, 3, 4, 5, 6, 7, 8, 12, 15, 16, 17])
        assert g.keys() == t.keys()
        for k in t:
            assert np.array_equal(g[k], t[k]), f"points of manifold {k} differ"
        assert started - seen == created
        seen = started
    w.close(); d.close()


def test_device_binding_follows_the_real_cpu_stepper(dev, E, O):
    """Same user code, the reference's stepper_sequential on the CPU and stepper_b2d on the GPU: identical in free fall
    (no row order involved; sinf / cosf may differ from glibc by an ulp), the same resting pile afterwards."""
    if O.ref_stepper() is None:
        pytest.skip("oracle/_ref/libedyn_stepper.so not shipped")
    scene = G.build_scene(E, "boxes_27")
    st = scene["settings"]
    w = EdynB2dWorld(O, dev, scene, max_manifolds=MAX_MANIFOLDS)
    r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    G.populate(r, scene)
    w.step(5); r.step(5)
    a, b = w.state(), r.state()
    for k in ("pos", "orn", "linvel", "angvel"):
        assert np.abs(a[k] - b[k]).max() <= 1e-6, k
    w.step(175); r.step(175)
    a, b = w.state(), r.state()
    assert np.abs(a["pos"] - b["pos"]).max() < 1e-2 and np.abs(a["linvel"]).max() < 0.05
    w.close()


def test_device_chains_follow_the_real_stepper_free_running(gpu, E):
    """No oracle in between: the B200 and the reference's real stepper_sequential (its end state recorded by
    tests/golden/make_ref_runs.py), both free-running for 1000 steps on a slice of config 5 (64 chains): the hinge-chain
    family is insensitive to the sweep order, so north_star's 1e-4 must simply hold (5e-10 absolute under the CPU
    emulation of the kernels after 300 steps)."""
    runs = np.load(R.OUT)
    scene = E.scenes.hinge_chains(8, 8)
    w = E.scenes.build_world(scene)
    n = scene["dynamic"]
    w.step(1000)
    g, c = w.download_state(aabb=False), {k: runs[f"chains_8x8.1000.{k}"] for k in ("pos", "linvel")}
    rel = float(np.abs(g["pos"][:n] - c["pos"]).max() / np.abs(c["pos"]).max())
    assert rel <= 1e-4, f"relative position error after 1000 steps {rel:.3e}"
    assert float(np.abs(g["linvel"][:n] - c["linvel"]).max()) <= 1e-3
    w.close()


@pytest.mark.xfail(strict=False, reason="first run on hardware: the restitution solver was written after the round's GPU budget ended and is "
                                        "verified under the CPU emulation only (tests/test_emu_device.py::test_emulated_restitution_solver)")
def test_device_restitution_solver_matches_oracle(gpu, E, O):
    """B2D_FLAG_RESTITUTION_SOLVER on the B200 in lock step with the oracle's restatement of restitution_solver.cpp (the
    reference's default settings), mixed pile with e = 0.2 and a random scene with e up to 0.8."""
    from tests.emu.lockstep import lockstep
    from tests.test_ref_stepper import random_scene
    for scene in (E.scenes.mixed_pile(5, jitter=0.01), random_scene(E, O, 3)):
        res = lockstep(E, O, scene, 100, restitution_solver=True)
        assert res["ok"] and res["worst"] <= 1e-5, (scene["name"], res)
