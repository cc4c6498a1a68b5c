"""GPU tests of the pieces the multi-GPU path adds: body removal (registry.destroy) against the oracle through the C
ABI, and -- on a box with at least two GPUs -- island migration between two ranks over NCCL (SURVEY.md section 8e)."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
f32 = np.float32


def _make_oracle(O, scene):
    o = O.OracleWorld(vel_iters=scene["settings"]["velocity_iterations"], pos_iters=scene["settings"]["position_iterations"])
    o.add_bodies(scene["bodies"])
    if scene["hinges"]:
        h = scene["hinges"]
        o.add_hinges(h["a"], h["b"], h["pivot_a"], h["pivot_b"], h["axis_a"], h["axis_b"])
    if scene["exclusions"] is not None:
        o.add_exclusions(*scene["exclusions"])
    return o


def _pairset(p):
    return {tuple(x) for x in p.tolist()}


@pytest.mark.parametrize("name", ["boxes", "chains"])
def test_remove_bodies_matches_oracle(gpu, E, O, name):
    """b2d_remove_bodies == registry.destroy: the bodies' manifolds and joints vanish, everything else carries on, and
    the device stays in lock step with the oracle (same check as test_lockstep_phase_parity) across the removal."""
    scene = E.scenes.boxes_on_plane(3, jitter=0.01) if name == "boxes" else E.scenes.hinge_chains(3, 4)
    w = E.scenes.build_world(scene)
    o = _make_oracle(O, scene)
    n = scene["dynamic"]
    gone = np.array([1, 4, 5, n - 1], np.uint32)
    for s in range(60):
        if s == 25:
            w.remove_bodies(gone); o.remove_bodies(gone)
        w.run_phases(E.world.PH_BROAD); o.run_phases(O.PH_BROAD)
        gp = _pairset(w.pairs())
        assert gp == _pairset(o.pairs()), f"step {s}: broadphase pair lists differ"
        if s >= 25:
            assert not any(a in gone or b in gone for a, b in gp), "a removed body still owns a manifold"
        w.run_phases(E.world.PH_NARROW | E.world.PH_ISLANDS); o.run_phases(O.PH_NARROW | O.PH_ISLANDS)
        gi, oi = w.islands(), o.islands()
        assert np.array_equal(gi, oi), f"step {s}: island partition differs"
        w.run_phases(E.world.PH_SOLVE)
        hi, pr = w.solver_order()
        o.set_order(hi, pr)
        o.run_phases(O.PH_SOLVE)
        g, c = w.download_state(), o.state()
        live = np.ones(len(g["pos"]), bool)
        if s >= 25:
            live[gone] = False
        for k in ("pos", "orn", "linvel", "angvel"):
            assert np.abs(g[k][live] - c[k][live]).max() <= 1e-5, f"step {s}: {k}"
        o.set_state(g["pos"], g["orn"], g["linvel"], g["angvel"])
        gc = w.contacts()
        o.set_contacts(gc["pairs"], gc["num"], gc["pts"], gc["att"], gc["lifetime"])
    assert w.stats()["error_flags"] == 0
    st = w.download_state()
    assert np.all(st["linvel"][gone] == 0), "a destroyed body no longer moves"


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _migration_worker(rank, world_size, port, q):
    import torch
    import torch.distributed as dist_mod
    import edyn_b200 as E
    from edyn_b200 import dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist_mod.init_process_group("nccl", rank=rank, world_size=world_size, device_id=torch.device("cuda", rank))
    import traceback
    try:
        scene = E.scenes.approaching_stacks(height=3, gap=0.6, speed=3.0)
        sw = dist.ShardedWorld(scene, rank, world_size, dist_mod, device=rank)
        first_hit = None
        for k in range(60):
            pairs = sw.step(1)
            if pairs and first_hit is None:
                first_hit = k
        st = sw.world.download_state()
        gids = np.asarray(sw.global_of_local)[sw.dynamic_local]
        q.put((rank, first_hit, sw.migrated_in, sw.migrated_out, gids.tolist(), st["pos"][sw.dynamic_local].tolist(),
               len(sw.world.pairs()), sw.world.stats()["error_flags"]))
    except Exception:
        # report instead of leaving the peer blocked in a collective until its timeout
        q.put((rank, "error", traceback.format_exc()))
        os._exit(1)
    finally:
        dist_mod.destroy_process_group()


def test_island_migration_two_gpus(gpu, E):
    """Two stacks owned by two GPUs slide into each other; rank 1 hands its island to rank 0 over NCCL, and the merged
    world tracks a single-GPU run of the whole scene."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_migration_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    try:
        for _ in procs:
            r = q.get(timeout=90)
            assert r[1] != "error", r[2]
            res.append(r)
    finally:
        for p in procs:
            p.join(timeout=20)
            if p.is_alive():
                p.kill()
    res.sort()
    assert all(p.exitcode == 0 for p in procs)
    (_, hit0, in0, out0, gid0, pos0, np0, err0), (_, hit1, in1, out1, gid1, pos1, np1, err1) = res
    assert hit0 == hit1 and hit0 is not None and hit0 > 0
    assert (in0, out0, in1, out1) == (3, 0, 0, 3)
    assert sorted(gid0) == list(range(6)) and gid1 == [] and np1 == 0 and err0 == err1 == 0
    scene = E.scenes.approaching_stacks(height=3, gap=0.6, speed=3.0)
    ref = E.scenes.build_world(scene)
    ref.step(60)
    want = ref.download_state()["pos"][:6]
    got = np.zeros((6, 3), f32)
    got[np.asarray(gid0)] = np.asarray(pos0, f32)
    # body ids (hence pair and Gauss-Seidel order) differ after the move: solver-tolerance agreement, not bitwise
    assert np.abs(got - want).max() < 5e-3, np.abs(got - want).max()


SLEEP_SCENES = {
    "sleep_and_wake": (lambda E: E.scenes.sleep_and_wake(), 400),
    "boxes_27": (lambda E: E.scenes.boxes_on_plane(3, jitter=0.01), 190),
    "approaching_stacks": (lambda E: E.scenes.approaching_stacks(height=2), 240),
}


@pytest.mark.parametrize("name", list(SLEEP_SCENES))
def test_island_sleeping_matches_oracle(gpu, E, O, name):
    """B2D_FLAG_SLEEPING: sleep timestamps, put_to_sleep and wake-up on the device in lock step with the oracle's
    restatement of island_manager.cpp:524-623 -- sleeping flags, pair lists, islands and state every step."""
    make, steps = SLEEP_SCENES[name]
    scene = make(E)
    w = E.scenes.build_world(scene, flags=E.world.FLAG_SLEEPING)
    o = _make_oracle(O, scene)
    o.set_sleeping(True)
    n = scene["dynamic"]
    slept = woke = 0
    prev = np.zeros(n, bool)
    for s in range(steps):
        w.run_phases(E.world.PH_BROAD); o.run_phases(O.PH_BROAD)
        assert _pairset(w.pairs()) == _pairset(o.pairs()), f"step {s}: broadphase pair lists differ"
        w.run_phases(E.world.PH_NARROW | E.world.PH_ISLANDS); o.run_phases(O.PH_NARROW | O.PH_ISLANDS)
        assert np.array_equal(w.islands(), o.islands()), f"step {s}: island partition differs"
        gs, os_ = w.sleeping(), o.sleeping()
        assert np.array_equal(gs, os_), f"step {s}: sleeping flags differ: {np.where(gs != os_)[0][:8]}"
        slept += int((gs[:n] & ~prev).sum()); woke += int((~gs[:n] & prev).sum()); prev = gs[:n].copy()
        w.run_phases(E.world.PH_SOLVE)
        hi, pr = w.solver_order()
        o.set_order(hi, pr)
        o.run_phases(O.PH_SOLVE)
        g, c = w.download_state(), o.state()
        for k in ("pos", "orn", "linvel", "angvel"):
            assert np.abs(g[k] - c[k]).max() <= 1e-5, f"step {s}: {k}"
        o.set_state(g["pos"], g["orn"], g["linvel"], g["angvel"])
        gc = w.contacts()
        o.set_contacts(gc["pairs"], gc["num"], gc["pts"], gc["att"], gc["lifetime"])
    assert w.stats()["error_flags"] == 0
    assert slept >= (3 if name == "sleep_and_wake" else n), f"{name}: only {slept} fall-asleep events"
    if name == "sleep_and_wake":
        assert woke == 1
    # wake_up_entity
    w.wake_bodies([0]); o.wake_bodies([0])
    w.run_phases(E.world.PH_ISLANDS); o.run_phases(O.PH_ISLANDS)
    assert np.array_equal(w.sleeping(), o.sleeping()) and not w.sleeping()[0]


def test_collision_exclusion_add_remove_clear_device(gpu, E, O):
    """test/edyn/collision/test_exclusion.cpp on the device path: b2d_add_exclusions / b2d_remove_exclusions and the
    edyn-style wrappers change which pairs the broadphase makes, identically to the oracle."""
    from edyn_b200.rigidbody import RigidBodyDef, bodies_soa, box_shape
    soa = bodies_soa([RigidBodyDef(position=(0.1 * i, 0, 0), mass=1.0, shape=box_shape((0.2, 0.2, 0.2))) for i in range(3)], (0.0, 0.0, 0.0))

    def run(ops):
        w = E.World(3, max_manifolds=64); w.add_bodies(soa)
        o = O.OracleWorld(); o.add_bodies(soa)
        for op, a, b in ops:
            if op == "+":
                E.exclude_collision(w, a, b); o.add_exclusions([a], [b])
            elif op == "-":
                E.remove_collision_exclusion(w, a, b); o.remove_exclusions([a], [b])
            else:
                gone = [p for p in w.exclusions if a in p]
                E.clear_collision_exclusion(w, a)
                for p in gone:
                    o.remove_exclusions([p[0]], [p[1]])
        w.run_phases(E.world.PH_BROAD); o.run_phases(O.PH_BROAD)
        got = _pairset(w.pairs())
        assert got == _pairset(o.pairs())
        return {tuple(sorted(p)) for p in got}
    assert run([]) == {(0, 1), (0, 2), (1, 2)}
    assert run([("+", 0, 1), ("+", 0, 2)]) == {(1, 2)}
    assert run([("+", 0, 1), ("+", 0, 2), ("-", 1, 0)]) == {(0, 1), (1, 2)}
    assert run([("+", 0, 1), ("+", 0, 2), ("+", 1, 2), ("clear", 0, 0)]) == {(0, 1), (0, 2)}


def test_issue_76_destroy_then_recreate_device(gpu, E):
    """test/edyn/issues/issue76.cpp through the C ABI: static floor made, destroyed, made again, stepped."""
    from edyn_b200.rigidbody import RigidBodyDef, box_shape, plane_shape
    w = E.attach(max_bodies=8, max_manifolds=64)
    floor_def = RigidBodyDef(kind=E.STATIC, shape=plane_shape((0, 1, 0), 0.0))
    f0 = E.make_rigidbody(w, floor_def)
    w.remove_bodies([f0])
    box = E.make_rigidbody(w, RigidBodyDef(position=(0, 0.5, 0), mass=1.0, shape=box_shape((0.5, 0.5, 0.5))))
    w.step(30)
    assert w.download_state()["pos"][box, 1] < 0.0 and len(w.pairs()) == 0, "the destroyed floor holds nothing up"
    f1 = E.make_rigidbody(w, floor_def)
    st = w.download_state()
    pos = st["pos"].copy(); pos[box] = (0, 0.5, 0)
    w.upload_state(pos, st["orn"], np.zeros_like(st["linvel"]), np.zeros_like(st["angvel"]))
    w.step(30)
    assert abs(w.download_state()["pos"][box, 1] - 0.5) < 1e-3
    assert _pairset(w.pairs()) == {(box, f1)}
    assert w.stats()["error_flags"] == 0
