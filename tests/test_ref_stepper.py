"""The oracle against the reference's REAL whole-step code.

oracle/_ref/libedyn_stepper.so is every translation unit of /root/reference/src/edyn (minus networking) compiled unmodified
against oracle/entt_lite, the functional stand-in for the absent EnTT dependency; oracle/ref_stepper.cpp drives
edyn::attach / make_rigidbody / make_constraint<hinge_constraint> / exclude_collision / edyn::step_simulation
(stepper_sequential.cpp:71-102).  The only thing the oracle takes from the reference is the ORDER in which the island
solver swept the rows that step (island_solver.cpp:181-222 walks island.edges, a sparse set filled by entity_graph
traversals); broadphase, narrowphase incl. contact persistence, islands, row preparation, warm starting, velocity and
position iterations, integration and the AABB / inertia refresh are all the oracle's own -- and must agree BIT FOR BIT.

  * live lock-step (needs the library: built by `make -C oracle stepper` where the reference's sources are),
  * the same comparison against what the library produced, recorded in tests/golden/whole_step.npz and
    tests/golden/ref_runs.npz (always runs)."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.golden import make_ref_runs as R
from tests.golden import make_whole_step as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "whole_step.npz")


@pytest.fixture(scope="module")
def refstep(O):
    if O.ref_stepper() is None:
        pytest.skip("oracle/_ref/libedyn_stepper.so not available (needs /root/reference at build time)")
    return O


def _keys(p):
    p = np.asarray(p, np.uint64).reshape(-1, 2)
    return (p[:, 0] << np.uint64(32)) | p[:, 1]


def _oracle_step(O, o, hinge_order, contact_order):
    o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
    o.set_point_order(hinge_order, contact_order)
    o.run_phases(O.PH_SOLVE)


def _same_partition(a, b):
    pa = np.unique(np.stack([a.astype(np.int64), b.astype(np.int64)], 1), axis=0)
    return len(np.unique(pa[:, 0])) == len(pa) and len(np.unique(pa[:, 1])) == len(pa)


def test_entt_lite_semantics(tmp_path):
    """Pool order, view order, swap-and-pop, identifier recycling, signals, paged storage: oracle/entt_lite/selftest.cpp."""
    cxx = shutil.which("g++")
    assert cxx, "g++ is part of the image"
    exe = str(tmp_path / "entt_selftest")
    subprocess.run([cxx, "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "oracle", "entt_lite"), "-o", exe,
                    os.path.join(ROOT, "oracle", "entt_lite", "selftest.cpp")], check=True)
    out = subprocess.run([exe], capture_output=True, text=True)
    assert out.returncode == 0 and "entt_lite ok" in out.stdout, out.stdout + out.stderr


@pytest.mark.parametrize("name", list(G.SCENES))
def test_oracle_lockstep_with_real_stepper(O, E, name):
    """The real stepper's row order of every step (whole_step.npz) replayed by the oracle; after each step state, AABBs,
    manifold set (ordered pairs), point counts and island partition must be the real stepper's, compared through the
    per-step digests recorded by tests/golden/make_ref_runs.py."""
    g, runs = np.load(GOLDEN), np.load(R.OUT)
    oh, oc, hoff, coff = g[f"{name}.order_h"], g[f"{name}.order_c"], g[f"{name}.order_h_off"], g[f"{name}.order_c_off"]
    want = runs[f"{name}.digests"]
    scene = G.build_scene(E, name)
    st = scene["settings"]
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    G.populate(o, scene)
    o.set_position_type_order(contacts_first=True)       # this build of the reference is GCC's (see the random-scene test)
    touched = 0
    for s in range(R.LOCKSTEP_STEPS):
        _oracle_step(O, o, oh[hoff[s]:hoff[s + 1]], oc[coff[s]:coff[s + 1]])
        c = o.contacts()
        assert R.step_digest(o.state(), c, o.islands()) == want[s], \
            f"{name} step {s}: state, AABBs, manifold set, point counts or island partition differ from the real stepper's"
        touched = max(touched, int(c["num"].sum()))
    assert touched > 0                                   # the scene did come to rest on its contacts
    # make_rigidbody derives the inverse inertia from mass and shape (dynamics/moment_of_inertia.cpp); the scene generators
    # (edyn_b200/rigidbody.py) must hand the device the same numbers
    dyn = np.asarray(scene["bodies"]["kind"]) == 0
    assert np.array_equal(runs[f"{name}.inertia_inv"][dyn], np.asarray(scene["bodies"]["inv_inertia"], np.float32).reshape(-1, 9)[dyn])


# ----------------------------------------------------------------------------- random scenes

def _unit_quat(rng, fixed_point, fns):
    """Random orientation.  fixed_point: one that normalize() maps to itself bit for bit -- position_solver::solve
    normalises the orientation of BOTH bodies in place, a static one included (position_solver.hpp:26-32), which moves a
    quaternion that is an ulp off unit length; oracle and device leave non-procedural bodies alone."""
    while True:
        q = rng.normal(size=4)
        q = (q / np.linalg.norm(q)).astype(np.float32)
        if not fixed_point or np.array_equal(q, np.asarray(fns.integrate(q, np.zeros(3, np.float32), 1 / 60), np.float32)):
            return tuple(q)


def random_scene(E, O, seed, n=40, kinematic=2, hinges=4, statics=3):
    """n dynamic spheres / boxes / capsules of random size, pose, velocity, mass, friction and restitution (0, 0.3, 0.8:
    through the row rhs), a third of them with collision filters, kinematic platforms moving and turning, arbitrarily
    oriented static boxes, a ground plane, hinges between random pairs with arbitrary pivots (two of them excluded from
    colliding) -- so joints and contacts act on the same bodies."""
    R = E.rigidbody
    rng, fns = np.random.default_rng(seed), O.ora_fns()
    defs = []
    for _ in range(n):
        shape = [R.sphere_shape(float(rng.uniform(0.15, 0.4))), R.box_shape(tuple(rng.uniform(0.12, 0.45, 3))),
                 R.capsule_shape(float(rng.uniform(0.1, 0.25)), float(rng.uniform(0.1, 0.4)), int(rng.integers(3)))][rng.integers(3)]
        d = R.RigidBodyDef(position=tuple(rng.uniform([-1.5, 0.5, -1.5], [1.5, 4.0, 1.5])), orientation=_unit_quat(rng, False, fns),
                           mass=float(rng.choice([0.5, 1.0, 2.0, 4.0, 8.0])),          # 1 / (1 / m) == m: the harness hands inv_mass over
                           linvel=tuple(rng.uniform(-2, 2, 3)), angvel=tuple(rng.uniform(-3, 3, 3)), shape=shape,
                           material=R.Material(restitution=float(rng.choice([0, 0.3, 0.8])), friction=float(rng.uniform(0.1, 1.0))))
        if rng.random() < 0.3:
            d.collision_group, d.collision_mask = int(rng.choice([1, 2, 4])), int(rng.choice([1, 3, 6, 7]))
        defs.append(d)
    for _ in range(kinematic):
        defs.append(R.RigidBodyDef(kind=R.KINEMATIC, position=(float(rng.uniform(-1, 1)), 0.4, float(rng.uniform(-1, 1))),
                                   linvel=(float(rng.uniform(-0.5, 0.5)), 0, float(rng.uniform(-0.5, 0.5))),
                                   angvel=(0, float(rng.uniform(-1, 1)), 0), shape=R.box_shape((0.5, 0.2, 0.5))))
    for _ in range(statics):
        defs.append(R.RigidBodyDef(kind=R.STATIC, position=tuple(rng.uniform([-2, 0.2, -2], [2, 0.6, 2])),
                                   orientation=_unit_quat(rng, True, fns), shape=R.box_shape((0.4, 0.3, 0.4))))
    defs.append(R.RigidBodyDef(kind=R.STATIC, shape=R.plane_shape((0, 1, 0), 0.0)))
    f = np.float32
    a = rng.choice(n, size=hinges, replace=False).astype(np.uint32)
    b = ((a + 1 + rng.integers(n - 1, size=hinges)) % n).astype(np.uint32)
    hs = dict(a=a, b=b, pivot_a=rng.uniform(-0.3, 0.3, (hinges, 3)).astype(f), pivot_b=rng.uniform(-0.3, 0.3, (hinges, 3)).astype(f),
              axis_a=np.tile(np.array([0, 0, 1], f), (hinges, 1)), axis_b=np.tile(np.array([0, 1, 0], f), (hinges, 1)))
    return dict(name=f"random_{seed}", bodies=R.bodies_soa(defs), hinges=hs, exclusions=(a[:2].copy(), b[:2].copy()), dynamic=n,
                settings=dict(velocity_iterations=10, position_iterations=3))


def random_scene_wide(E, O, seed):
    """Wider than random_scene: 8-90 bodies, masses 0.25-16, friction 0-2, restitution up to 1, some bodies with their own
    gravity, kinematic boxes / spheres / capsules moving in all directions, static boxes / spheres / capsules, the ground
    a level plane, a TILTED plane or a big static box, hinges with random axes on both sides, 1-20 velocity and 0-6
    position iterations."""
    R = E.rigidbody
    rng, fns = np.random.default_rng(10_000 + seed), O.ora_fns()
    n, ext = int(rng.integers(8, 90)), float(rng.uniform(0.8, 2.5))
    kinematic, statics = int(rng.integers(0, 4)), int(rng.integers(0, 6))
    hinges = int(rng.integers(0, min(8, n // 2)))
    defs = []
    for _ in range(n):
        shape = [R.sphere_shape(float(rng.uniform(0.1, 0.5))), R.box_shape(tuple(rng.uniform(0.08, 0.6, 3))),
                 R.capsule_shape(float(rng.uniform(0.08, 0.3)), float(rng.uniform(0.05, 0.5)), int(rng.integers(3)))][rng.integers(3)]
        d = R.RigidBodyDef(position=tuple(rng.uniform([-ext, 0.3, -ext], [ext, 5.0, ext])), orientation=_unit_quat(rng, False, fns),
                           mass=float(rng.choice([0.25, 0.5, 1.0, 2.0, 4.0, 8.0, 16.0])), linvel=tuple(rng.uniform(-4, 4, 3)),
                           angvel=tuple(rng.uniform(-6, 6, 3)), shape=shape,
                           material=R.Material(restitution=float(rng.choice([0, 0, 0.3, 0.8, 1.0])), friction=float(rng.choice([0.0, 0.1, 0.5, 1.0, 2.0]))))
        if rng.random() < 0.3:
            d.collision_group, d.collision_mask = int(rng.choice([1, 2, 4])), int(rng.choice([1, 3, 6, 7]))
        if rng.random() < 0.1:
            d.gravity = tuple(rng.uniform(-3, 3, 3))
        defs.append(d)
    for _ in range(kinematic):
        defs.append(R.RigidBodyDef(kind=R.KINEMATIC, position=tuple(rng.uniform([-1, 0.2, -1], [1, 1.5, 1])), linvel=tuple(rng.uniform(-1, 1, 3)),
                                   angvel=tuple(rng.uniform(-2, 2, 3)),
                                   shape=[R.box_shape((0.5, 0.2, 0.5)), R.sphere_shape(0.4), R.capsule_shape(0.2, 0.5, 0)][rng.integers(3)]))
    for _ in range(statics):
        defs.append(R.RigidBodyDef(kind=R.STATIC, position=tuple(rng.uniform([-2, 0.1, -2], [2, 1.0, 2])), orientation=_unit_quat(rng, True, fns),
                                   shape=[R.box_shape(tuple(rng.uniform(0.2, 0.8, 3))), R.sphere_shape(float(rng.uniform(0.2, 0.6))),
                                          R.capsule_shape(0.2, 0.6, int(rng.integers(3)))][rng.integers(3)]))
    ground = rng.integers(3)          # planes through the origin: collide_sphere_plane.cpp:17 mis-places pivotB by 2 n c otherwise (DESIGN.md section 6)
    if ground == 0:
        defs.append(R.RigidBodyDef(kind=R.STATIC, shape=R.plane_shape((0, 1, 0), 0.0)))
    elif ground == 1:
        nrm = np.array([rng.uniform(-0.2, 0.2), 1.0, rng.uniform(-0.2, 0.2)])
        nrm = (nrm / np.linalg.norm(nrm)).astype(np.float32)
        defs.append(R.RigidBodyDef(kind=R.STATIC, shape=R.plane_shape(tuple(float(x) for x in nrm), 0.0)))
    else:
        defs.append(R.RigidBodyDef(kind=R.STATIC, position=(0, -1.0, 0), shape=R.box_shape((6.0, 1.0, 6.0))))
    f, hs, ex = np.float32, None, None
    if hinges:
        a = rng.choice(n, size=hinges, replace=False).astype(np.uint32)
        b = ((a + 1 + rng.integers(n - 1, size=hinges)) % n).astype(np.uint32)
        ax, bx = rng.normal(size=(hinges, 3)), rng.normal(size=(hinges, 3))
        ax, bx = (ax / np.linalg.norm(ax, axis=1, keepdims=True)).astype(f), (bx / np.linalg.norm(bx, axis=1, keepdims=True)).astype(f)
        hs = dict(a=a, b=b, pivot_a=rng.uniform(-0.4, 0.4, (hinges, 3)).astype(f), pivot_b=rng.uniform(-0.4, 0.4, (hinges, 3)).astype(f), axis_a=ax, axis_b=bx)
        k = int(rng.integers(0, hinges + 1))
        ex = (a[:k].copy(), b[:k].copy()) if k else None
    return dict(name=f"wide_{seed}", bodies=R.bodies_soa(defs), hinges=hs, exclusions=ex, dynamic=n,
                settings=dict(velocity_iterations=int(rng.choice([1, 4, 8, 20])), position_iterations=int(rng.choice([0, 1, 3, 6]))))


def _refines(fine, coarse):
    pa = np.unique(np.stack([coarse.astype(np.int64), fine.astype(np.int64)], 1), axis=0)
    return len(np.unique(pa[:, 1])) == len(pa), len(np.unique(pa[:, 0])) == len(pa)


@pytest.mark.parametrize("seeds", [range(0, 12), range(12, 24), range(24, 40)])
def test_random_scenes_lockstep_with_real_stepper(refstep, E, seeds):
    """150 free-running steps of 46-body random scenes: state and AABBs bit-identical, manifold sets (ordered pairs) and
    point counts identical, every step.  Beyond the row order two more things follow this build of the reference:
      * the position iterations sweep contacts BEFORE joints: island_solver.cpp:340 expands the constraint types as
        arguments of max_variadic(...), so the type order is the compiler's argument evaluation order (GCC: right to left;
        tuple order -- joints first -- is what oracle and device do by default);
      * the island BOOKKEEPING: a split pending on an island is lost when that island is merged into a bigger one in the
        same step (island_manager.cpp:352-357 after :297-350), so the reference's partition can be coarser than the
        connected components for a while (seed 36); it only shows in the per-island position-iteration early-out.  The
        oracle's own partition must always REFINE the reference's, and is replaced by it before the solve."""
    O = refstep
    coarser = 0
    for seed in seeds:
        scene = random_scene(E, O, seed)
        st = scene["settings"]
        r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
        o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
        G.populate(r, scene); G.populate(o, scene)
        o.set_position_type_order(contacts_first=True)
        dyn = np.asarray(scene["bodies"]["kind"]) == 0
        for s in range(150):
            r.step(1)
            hi, ct = r.solver_order()
            o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
            ref_islands = r.islands()
            refines, equal = _refines(o.islands()[dyn], ref_islands[dyn])
            assert refines, f"seed {seed} step {s}: the oracle's islands are not a refinement of the reference's"
            coarser += not equal
            o.set_islands(ref_islands)
            o.set_point_order(hi, ct)
            o.run_phases(O.PH_SOLVE)
            a, b = r.state(), o.state()
            for k in ("pos", "orn", "linvel", "angvel", "aabb"):
                assert np.array_equal(a[k], b[k]), f"seed {seed} step {s}: {k} differs by {np.abs(a[k] - b[k]).max():.3e}"
            rc, oc = r.contacts(), o.contacts()
            ri, oi = np.argsort(_keys(rc["pairs"])), np.argsort(_keys(oc["pairs"]))
            assert np.array_equal(_keys(rc["pairs"])[ri], _keys(oc["pairs"])[oi]), f"seed {seed} step {s}: manifold sets differ"
            assert np.array_equal(rc["num"][ri], oc["num"][oi]), f"seed {seed} step {s}: point counts differ"
    assert coarser <= 15 * len(seeds)            # the lagging bookkeeping is the exception, not the rule


MEDIUM = {
    "boxes_512": (lambda E: E.scenes.boxes_on_plane(8), 90),
    "mixed_1000": (lambda E: E.scenes.mixed_pile(10), 90),
    "spheres_2048": (lambda E: E.scenes.spheres_in_box(16, 8, 16), 90),
    "chains_4096": (lambda E: E.scenes.hinge_chains(32, 32), 40),
}


def lockstep(O, scene, steps, threads=1, restitution_iterations=0):
    """Free-running lock step of the real stepper and the oracle (row order and island bookkeeping follow the reference);
    returns (first step with any difference or None, steps on which the reference's partition was coarser, contact points).
    restitution_iterations > 0: the restitution solver runs on both sides (settings.num_restitution_iterations; the
    reference's default is 8); it walks the entity graph breadth first, so the graph's adjacency order and island.edges
    order at the start of solver::update are handed to the oracle as well (refs_get_graph_order)."""
    st = scene["settings"]
    r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"], restitution_iters=restitution_iterations)
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"], threads=threads)
    G.populate(r, scene); G.populate(o, scene)
    o.set_position_type_order(contacts_first=True)
    o.set_restitution_iterations(restitution_iterations)
    dyn = np.asarray(scene["bodies"]["kind"]) == 0
    first_bad, coarser, points = None, 0, 0
    for s in range(steps):
        if restitution_iterations:
            r.step_begin()                               # broadphase, narrowphase, island manager
            graph = r.graph_order()
            r.step_end()                                 # solver::update: restitution solver first, then the rest
        else:
            r.step(1)
        hi, ct = r.solver_order()
        o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
        ref_islands = r.islands()
        refines, equal = _refines(o.islands()[dyn], ref_islands[dyn])
        assert refines, f"step {s}: the oracle's islands are not a refinement of the reference's"
        coarser += not equal
        o.set_islands(ref_islands)
        o.set_point_order(hi, ct)
        if restitution_iterations:
            o.set_graph_order(*graph)
        o.run_phases(O.PH_SOLVE)
        a, b = r.state(), o.state()
        rc, oc = r.contacts(), o.contacts()
        same = all(np.array_equal(a[k], b[k]) for k in ("pos", "orn", "linvel", "angvel", "aabb")) and \
            np.array_equal(np.sort(_keys(rc["pairs"])), np.sort(_keys(oc["pairs"]))) and int(rc["num"].sum()) == int(oc["num"].sum())
        if not same and first_bad is None:
            first_bad = s
        points = int(rc["num"].sum())
    return first_bad, coarser, points


@pytest.mark.parametrize("name", list(MEDIUM))
def test_oracle_lockstep_with_real_stepper_medium_scenes(refstep, E, name):
    """Hundreds to thousands of bodies, thousands of contact points, the oracle on all host threads (its per-island solve
    is threaded like run_island_solver_seq_mt): still bit for bit.  tools/ref_lockstep.py runs the same at benchmark sizes
    (config 2 and config 3 at full size, 1/16 of config 5, 1/64 of config 4); results in DESIGN.md section 6."""
    make, steps = MEDIUM[name]
    first_bad, _, points = lockstep(refstep, make(E), steps, threads=os.cpu_count() or 1)
    assert first_bad is None, f"{name}: first difference at step {first_bad}"
    assert points > 1000


SLEEPY = {
    "sleep_and_wake": (lambda E: E.scenes.sleep_and_wake(), 500, 3),        # sleeps, is woken by an impact, both sleep again
    "boxes_27": (lambda E: E.scenes.boxes_on_plane(3), 400, 1),
    "approaching_stacks": (lambda E: E.scenes.approaching_stacks(), 500, 1),
}


@pytest.mark.parametrize("name", list(SLEEPY))
def test_island_sleeping_matches_real_stepper(refstep, E, name):
    """Bodies created WITHOUT sleeping_disabled: island sleep timestamps, put_to_sleep after island_time_to_sleep = 2 s,
    wake-up when a new edge joins a sleeping island (island_manager.cpp:257-295, :541-623) -- sleeping_tag per body and the
    whole state identical to the restatement's every step.  Step j is given the time stepper_sequential::update gives it
    (j * fixed_dt from attach time 0), which is also the restatement's and the device's clock."""
    O = refstep
    make, steps, min_events = SLEEPY[name]
    scene = make(E)
    st = scene["settings"]
    r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    r.add_bodies(scene["bodies"], sleeping_disabled=False)
    o.add_bodies(scene["bodies"])
    o.set_sleeping(True)
    o.set_position_type_order(contacts_first=True)
    events, prev = 0, np.zeros(len(scene["bodies"]["kind"]), bool)
    for s in range(steps):
        r.step(1)
        hi, ct = r.solver_order()
        _oracle_step(O, o, hi, ct)
        asleep = r.sleeping()
        assert np.array_equal(asleep, o.sleeping().astype(bool)), f"{name} step {s}: sleeping flags differ"
        a, b = r.state(), o.state()
        for k in ("pos", "orn", "linvel", "angvel"):
            assert np.array_equal(a[k], b[k]), f"{name} step {s}: {k} differs"
        events += not np.array_equal(asleep, prev)
        prev = asleep
    assert events >= min_events and prev.any()


@pytest.mark.parametrize("seeds", [range(0, 20), range(20, 40)])
def test_wide_random_scenes_lockstep_with_real_stepper(refstep, E, seeds):
    """random_scene_wide, 150 free-running steps each (120 seeds x 200 steps were run while writing this: all identical)."""
    for seed in seeds:
        first_bad, _, _ = lockstep(refstep, random_scene_wide(E, refstep, seed), 150)
        assert first_bad is None, f"seed {seed}: first difference at step {first_bad}"


def _lockstep_with_mutations(O, scene, steps, seed):
    from edyn_b200 import rigidbody as E_rigidbody
    """Every 17th step user code interferes: registry.destroy(body), remove_collision_exclusion, a patched velocity, or
    make_rigidbody of a new body (which recycles the identifier of a destroyed entity)."""
    rng = np.random.default_rng(seed)
    st = scene["settings"]
    r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    G.populate(r, scene); G.populate(o, scene)
    o.set_position_type_order(contacts_first=True)
    o.set_pool_order(True)               # destroying a body reorders the pool the broadphase iterates (swap and pop)
    kind = np.asarray(scene["bodies"]["kind"]).copy()
    alive = np.ones(len(kind), bool)
    excluded = list(zip(*[x.tolist() for x in scene["exclusions"]])) if scene["exclusions"] is not None else []
    events = 0
    for s in range(steps):
        if s and s % 17 == 0:
            what = rng.integers(4)
            movable = np.where(alive & (kind == 0))[0]
            if what == 0 and len(movable) > 4:
                b = int(rng.choice(movable))
                r.destroy_body(b); o.remove_bodies([b]); alive[b] = False
            elif what == 3:
                R = E_rigidbody
                d = R.RigidBodyDef(position=tuple(rng.uniform([-1, 2, -1], [1, 4, 1])), mass=float(rng.choice([0.5, 1.0, 2.0])),
                                   linvel=tuple(rng.uniform(-2, 2, 3)),
                                   shape=[R.sphere_shape(0.3), R.box_shape((0.3, 0.2, 0.25)), R.capsule_shape(0.15, 0.3, 1)][rng.integers(3)])
                soa = R.bodies_soa([d])
                r.add_bodies(soa); o.add_bodies(soa)
                kind, alive = np.append(kind, 0), np.append(alive, True)
            elif what == 1 and excluded:
                a, b = excluded.pop()
                if alive[a] and alive[b]:
                    r.remove_exclusion(a, b); o.remove_exclusions([a], [b])
            else:
                b = int(rng.choice(movable))
                lv, av = rng.uniform(-3, 3, 3).astype(np.float32), rng.uniform(-3, 3, 3).astype(np.float32)
                r.set_velocity(b, lv, av)
                x = o.state()
                x["linvel"][b], x["angvel"][b] = lv, av
                o.set_state(x["pos"], x["orn"], x["linvel"], x["angvel"])
            events += 1
        r.step(1)
        hi, ct = r.solver_order()
        o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
        dyn = (kind == 0) & alive
        ref_islands = r.islands()
        assert _refines(o.islands()[dyn], ref_islands[dyn])[0], f"step {s}: islands"
        o.set_islands(ref_islands)
        o.set_point_order(hi, ct)
        o.run_phases(O.PH_SOLVE)
        a, b = r.state(), o.state()
        for k in ("pos", "orn", "linvel", "angvel"):
            assert np.array_equal(a[k][alive], b[k][alive]), f"seed {seed} step {s}: {k}"
        rc, oc = r.contacts(), o.contacts()
        assert np.array_equal(np.sort(_keys(rc["pairs"])), np.sort(_keys(oc["pairs"]))), f"seed {seed} step {s}: manifold sets (ordered pairs)"
        assert int(rc["num"].sum()) == int(oc["num"].sum())
    return events


def test_user_code_between_steps_matches_real_stepper(refstep, E):
    """Bodies destroyed, exclusions removed and velocities patched while the simulation runs: the restatement follows the
    real stepper bit for bit (20 + 100 seeds were run; 12 here).  One more EnTT artefact shows here: registry.destroy(body)
    is a swap-and-pop in the procedural_tag pool, the newest body takes the removed one's place in the broadphase's
    iteration, and with it changes which body of a later pair becomes body[0].  The oracle reproduces that on request
    (set_pool_order); its default, and the device's rule, is descending body id -- after removals the device may therefore
    hold a manifold as (B, A) where this build of the reference holds (A, B)."""
    O = refstep
    events = 0
    for seed in range(6):
        events += _lockstep_with_mutations(O, random_scene(E, O, seed), 150, seed)
    for seed in range(6):
        events += _lockstep_with_mutations(O, random_scene_wide(E, O, seed), 200, seed)
    assert events > 80


def test_restitution_solver_matches_real_stepper(refstep, E):
    """The reference's DEFAULT settings (8 restitution iterations x 3 individual ones, restitution_solver.cpp:86-408):
    propagation of the bounce from the fastest penetrating manifold outwards, rows without restitution afterwards
    (solver.cpp:217-236) -- the restatement is bit-identical on the mixed pile (e = 0.2) and on random scenes with
    e in {0, 0.3, 0.8, 1}, and the solver does change the outcome (0.6 m after one second on seed 3)."""
    O = refstep
    assert lockstep(O, G.build_scene(E, "mixed_125"), 150, restitution_iterations=8)[0] is None
    for seed in range(8):
        assert lockstep(O, random_scene(E, O, seed), 150, restitution_iterations=8)[0] is None, f"seed {seed}"
    for seed in range(16):
        assert lockstep(O, random_scene_wide(E, O, seed), 150, restitution_iterations=8)[0] is None, f"wide seed {seed}"
    scene = random_scene(E, O, 3)
    st, ends = scene["settings"], []
    for iters in (0, 8):
        r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"], restitution_iters=iters)
        G.populate(r, scene)
        r.step(60)
        ends.append(r.state()["pos"])
    assert np.abs(ends[0] - ends[1]).max() > 0.1


def test_python_make_rigidbody_mirror_matches_real_make_rigidbody(E):
    """edyn_b200.rigidbody (what bench.py and the Python adapter stage) vs util/rigidbody.cpp:47-185 on 600 random bodies
    (recorded by tests/golden/make_ref_runs.py): inverse inertia of spheres / boxes / capsules (all three axes) identical
    to the last bit."""
    runs = np.load(R.OUT)
    soa = R.random_bodies(E)
    assert np.array_equal(runs["make_rigidbody.inertia_inv"], soa["inv_inertia"].reshape(-1, 9))
    assert np.array_equal(runs["make_rigidbody.aabb"][:, :3] <= runs["make_rigidbody.pos"], np.ones((600, 3), bool))


def test_real_stepper_multithreaded_matches_sequential(refstep, E):
    """execution_mode::sequential_multithreaded (what bench.py's reference arm times) gives the sequential mode's results."""
    O = refstep
    scene = G.build_scene(E, "mixed_125")
    st = scene["settings"]
    worlds = [O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"], threads=t) for t in (0, 4)]
    for w in worlds:
        G.populate(w, scene)
        w.step(60)
    a, b = worlds[0].state(), worlds[1].state()
    for k in ("pos", "orn", "linvel", "angvel"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("name", list(G.SCENES))
def test_oracle_replays_reference_trajectories(O, E, name):
    """Same comparison against the committed recording (tests/golden/make_whole_step.py): runs wherever the repo does."""
    g = np.load(GOLDEN)
    steps, keep = (int(v) for v in g["steps"])
    scene = G.build_scene(E, name)
    st = scene["settings"]
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    G.populate(o, scene)
    o.set_position_type_order(contacts_first=True)
    oh, oc, hoff, coff = g[f"{name}.order_h"], g[f"{name}.order_c"], g[f"{name}.order_h_off"], g[f"{name}.order_c_off"]
    for s in range(steps):
        _oracle_step(O, o, oh[hoff[s]:hoff[s + 1]], oc[coff[s]:coff[s + 1]])
        if (s + 1) % keep == 0:
            x = o.state()
            got = np.concatenate([x["pos"], x["orn"], x["linvel"], x["angvel"]], axis=1)
            want = g[f"{name}.states"][(s + 1) // keep - 1]
            assert np.array_equal(got, want), f"{name} step {s}: |oracle - reference| = {np.abs(got - want).max():.3e}"
    c = o.contacts()
    assert np.array_equal(np.sort(_keys(c["pairs"])), np.sort(_keys(g[f"{name}.final_pairs"])))
    assert int(c["num"].sum()) == int(g[f"{name}.final_num"].sum())
    assert _same_partition(o.islands(), g[f"{name}.islands"])
