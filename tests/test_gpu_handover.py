"""GPU tests of the device-resident multi-GPU path (SURVEY.md section 8e) and of the boundary pieces it leans on:
CUDA-graph replay of the step, dirty-subset staging (b2d_upload_bodies), kinematic bodies, collision filters, and the
island hand-over (b2d_island_halo / b2d_handover_plan / _pack / _unpack) driven by DeviceShardedWorld.

The hand-over is run twice: with ranks as THREADS sharing one device (always runs, so the driver's single-GPU box
exercises the same library code) and with one process per GPU over NCCL (needs >= 2 GPUs)."""
import os
import socket
import threading

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


# ----------------------------------------------------------------------------- CUDA graphs

@pytest.mark.parametrize("timing", [True, False])
def test_step_graphs_match_plain_launches(gpu, E, timing):
    """A step replayed from CUDA graphs (three segments with timing events, or one graph) leaves exactly the bits the
    plain launch sequence leaves."""
    scene = E.scenes.mixed_pile(6, jitter=0.01)
    os.environ["B2D_GRAPH"] = "0"
    try:
        plain = E.scenes.build_world(scene)
    finally:
        del os.environ["B2D_GRAPH"]
    graph = E.scenes.build_world(scene)
    graph.set_timing(timing)
    for _ in range(3):
        plain.step(20); graph.step(20)
        a, b = plain.download_state(), graph.download_state()
        for k in ("pos", "orn", "linvel", "angvel", "aabb"):
            assert np.array_equal(a[k], b[k]), k
    assert graph.stats()["kernel_launches"] == plain.stats()["kernel_launches"]
    assert graph.stats()["error_flags"] == 0


# ----------------------------------------------------------------------------- dirty-subset staging

def test_upload_bodies_equals_full_resync(gpu, E):
    """b2d_upload_bodies on a subset == b2d_upload_state with the same values written into the full arrays."""
    scene = E.scenes.mixed_pile(5, jitter=0.01)
    a, b = E.scenes.build_world(scene), E.scenes.build_world(scene)
    a.step(30); b.step(30)
    st = a.download_state(aabb=False)
    rng = np.random.default_rng(7)
    ids = rng.choice(scene["dynamic"], 17, replace=False).astype(np.uint32)
    st["pos"][ids] += rng.uniform(-0.05, 0.05, (17, 3)).astype(f32)
    st["linvel"][ids] = rng.uniform(-1, 1, (17, 3)).astype(f32)
    q = rng.normal(size=(17, 4)); q /= np.linalg.norm(q, axis=1, keepdims=True)
    st["orn"][ids] = q.astype(f32)
    a.upload_state(st["pos"], st["orn"], st["linvel"], st["angvel"])
    b.upload_bodies(ids, pos=st["pos"][ids], orn=st["orn"][ids], linvel=st["linvel"][ids])
    for _ in range(2):
        sa, sb = a.download_state(inv_IW=True), b.download_state(inv_IW=True)
        for k in ("pos", "orn", "linvel", "angvel", "aabb", "inv_IW"):
            assert np.array_equal(sa[k], sb[k]), k
        a.step(5); b.step(5)
    with pytest.raises(E.B2DError, match="range"):
        b.upload_bodies([10 ** 6], pos=np.zeros((1, 3), f32))


def test_material_and_mass_patch(gpu, E, O):
    """mass / inertia / material changes through the patch reach the next step exactly as if the body had been created
    with them (oracle built from the patched definition, lock step)."""
    scene = E.scenes.boxes_on_plane(2, jitter=0.01)
    w = E.scenes.build_world(scene)
    ids = np.array([1, 5], np.uint32)
    b = scene["bodies"]
    b["inv_mass"][ids] = f32(0.25); b["inv_inertia"][ids] *= f32(0.25); b["friction"][ids] = f32(0.1); b["restitution"][ids] = f32(0.3)
    w.upload_bodies(ids, inv_mass=b["inv_mass"][ids], inv_inertia=b["inv_inertia"][ids], friction=b["friction"][ids], restitution=b["restitution"][ids])
    o = _make_oracle(O, scene)
    _lockstep(E, O, w, o, 40)


def _pairset(p):
    return {tuple(x) for x in p.tolist()}


def _by_pair(c):
    return {tuple(p): k for k, p in enumerate(c["pairs"].tolist())}


def _lockstep(E, O, w, o, steps, before_step=None):
    for s in range(steps):
        if before_step:
            before_step(s)
        w.run_phases(E.world.PH_BROAD); o.run_phases(O.PH_BROAD)
        assert _pairset(w.pairs()) == _pairset(o.pairs()), f"step {s}: broadphase pair lists (body[0], body[1]) differ"
        w.run_phases(E.world.PH_NARROW | E.world.PH_ISLANDS); o.run_phases(O.PH_NARROW | O.PH_ISLANDS)
        assert np.array_equal(w.islands(), o.islands()), f"step {s}: island partition differs"
        gc, oc = w.contacts(), o.contacts()
        gi, oi = _by_pair(gc), _by_pair(oc)
        assert gi.keys() == oi.keys()
        for key, k in gi.items():
            j = oi[key]
            m = int(gc["num"][k])
            assert m == oc["num"][j] and np.array_equal(gc["att"][k, :m], oc["att"][j, :m]), f"step {s}: contact set differs for {key}"
        w.run_phases(E.world.PH_SOLVE)
        hi, pr = w.solver_order()
        o.set_order(hi, pr)
        o.run_phases(O.PH_SOLVE)
        g, c = w.download_state(), o.state()
        for k in ("pos", "orn", "linvel", "angvel"):
            assert np.abs(g[k] - c[k]).max() <= 1e-5, f"step {s}: {k} off by {np.abs(g[k] - c[k]).max()}"
        o.set_state(g["pos"], g["orn"], g["linvel"], g["angvel"])
        gc = w.contacts()
        o.set_contacts(gc["pairs"], gc["num"], gc["pts"], gc["att"], gc["lifetime"])
    assert w.stats()["error_flags"] == 0


def test_kinematic_body_pushes_a_stack(gpu, E, O):
    """constraint_body terms of a kinematic body (src/edyn/dynamics/solver.cpp:101-147): no mass, real velocity.  A
    kinematic slab slides under a stack of boxes; the host moves it every step through the patch call (that is what a
    user of kinematic bodies does), the device follows the oracle in lock step."""
    from edyn_b200.rigidbody import KINEMATIC
    scene = E.scenes.boxes_on_plane(2, jitter=0.0)
    b = scene["bodies"]
    slab = 0                                              # body 0 becomes a kinematic platform below the others
    b["kind"][slab] = KINEMATIC
    b["shape_params"][slab] = (3.0, 0.25, 3.0, 0)
    b["pos"][slab] = (0.5, 0.25, 0.5)
    b["pos"][1:8, 1] += 0.5
    b["inv_mass"][slab] = 0; b["inv_inertia"][slab] = 0; b["gravity"][slab] = 0
    b["linvel"][slab] = (0.6, 0, 0)
    w = E.scenes.build_world(scene)
    o = _make_oracle(O, scene)
    dt = f32(1.0 / 60)
    pos = b["pos"][slab].copy()

    def move(s):
        nonlocal pos
        if s == 0:
            return
        pos = (pos + b["linvel"][slab] * dt).astype(f32)
        w.upload_bodies([slab], pos=pos[None, :])
        st = o.state()
        st["pos"][slab] = pos
        o.set_state(st["pos"], st["orn"], st["linvel"], st["angvel"])
    _lockstep(E, O, w, o, 90, before_step=move)
    st = w.download_state()
    assert st["pos"][1:8, 0].mean() > 0.8, "friction against the moving platform carries the boxes along"
    assert np.all(st["linvel"][slab] == b["linvel"][slab])


def test_kind_patch_dynamic_to_kinematic(gpu, E, O):
    """Changing `kind` through the patch (dynamic -> kinematic) == creating the body kinematic."""
    from edyn_b200.rigidbody import KINEMATIC
    scene = E.scenes.boxes_on_plane(2, jitter=0.01)
    w = E.scenes.build_world(scene)
    b = scene["bodies"]
    b["kind"][3] = KINEMATIC; b["inv_mass"][3] = 0; b["inv_inertia"][3] = 0
    w.upload_bodies([3], kind=[KINEMATIC])
    o = _make_oracle(O, scene)
    _lockstep(E, O, w, o, 30)


def test_collision_filter_truth_table_device(gpu, E, O):
    """test/edyn/collision/test_broadphase.cpp:16-31 (should_collide_default's group / mask branch) on the device:
    overlapping boxes with every filter combination, pair list == oracle == the truth table."""
    from edyn_b200.rigidbody import RigidBodyDef, bodies_soa, box_shape
    cases = [  # (groupA, maskA, groupB, maskB, collide?)   None = no collision_filter component
        (1, 1, 1, 1, True), (1, 2, 2, 1, True), (1, 2, 1, 2, False), (1, 1, 2, 2, False), (3, 4, 4, 3, True),
        (None, None, 1, 1, True), (None, None, 0, 1, False), (None, None, 1, 0, False), (2, 2, None, None, True),
        (0xFFFFFFFFFFFFFFFF, 1, 1, 0x8000000000000000, True), (0x8000000000000000, 1, 2, 0x8000000000000000, False),
        (0x8000000000000000, 1, 1, 0x8000000000000000, True),
    ]
    for ga, ma, gb, mb, want in cases:
        defs = [RigidBodyDef(position=(0.0, 0, 0), mass=1.0, shape=box_shape((0.2, 0.2, 0.2))),
                RigidBodyDef(position=(0.1, 0, 0), mass=1.0, shape=box_shape((0.2, 0.2, 0.2)))]
        soa = bodies_soa(defs, (0.0, 0.0, 0.0))
        full = 0xFFFFFFFFFFFFFFFF
        soa["group"] = np.array([full if ga is None else ga, full if gb is None else gb], np.uint64)
        soa["mask"] = np.array([full if ma is None else ma, full if mb is None else mb], np.uint64)
        w = E.World(2, max_manifolds=16); w.add_bodies(soa)
        o = O.OracleWorld(); o.add_bodies(soa)
        w.run_phases(E.world.PH_BROAD); o.run_phases(O.PH_BROAD)
        assert _pairset(w.pairs()) == _pairset(o.pairs()), (ga, ma, gb, mb)
        assert (len(w.pairs()) == 1) == want, (ga, ma, gb, mb)


# ----------------------------------------------------------------------------- island hand-over

def _chains_scene(E):
    return E.scenes.hinge_chains(4, 6)           # 24 chains x 4 links; ranks split along x between chain columns 1 and 2


def _rank_body(rank, N, comm, scene_name, steps, q, device):
    import torch
    import edyn_b200 as E
    from edyn_b200 import dist
    torch.cuda.set_device(device)
    if scene_name == "stacks":
        scene = E.scenes.approaching_stacks(height=3, gap=0.6, speed=3.0)
    else:
        scene = _chains_scene(E)
    labels = dist.initial_islands(scene)
    sw = dist.DeviceShardedWorld(scene, rank, N, comm, device=device, labels=labels, slack=1.0)
    first_hit = None
    for k in range(steps):
        if scene_name == "chains" and k == 10 and rank == 1:
            # rank 1 shoves its first column of chains towards rank 0's last column
            ent = sw.world.entities()
            b = scene["bodies"]
            col = np.where((sw.owner[ent] == 1) & (b["pos"][ent, 0] < b["pos"][sw.owner == 1, 0].min() + 2.9))[0]
            v = np.zeros((len(col), 3), f32); v[:, 0] = -6.0
            sw.world.upload_bodies(col.astype(np.uint32), linvel=v)
        sw.step(1)
        if sw.halo_checks and first_hit is None:
            first_hit = k                        # first step whose rank boxes came within the broadphase margin
    w = sw.world
    st = w.download_state()
    ent = w.entities()
    alive = np.ones(w.num_bodies, bool)
    # bodies that left are removed slots: static, shapeless, at rest
    pr = w.pairs()
    hi, _ = w.solver_order()
    res = dict(rank=rank, first_hit=first_hit, migrated_in=sw.migrated_in, migrated_out=sw.migrated_out, dynamic=sw.dynamic,
               entities=ent.tolist(), pos=st["pos"].tolist(), linvel=st["linvel"].tolist(), pairs=ent[pr].tolist() if len(pr) else [],
               joints=int(len(hi)), err=w.stats()["error_flags"], rounds=sw.handover_rounds, bytes=comm.bytes_sent)
    q.append(res)
    sw.close()


def _run_threads(scene_name, steps):
    from edyn_b200 import dist
    shared = dist.ThreadComm.Shared(2)
    out, errs = [], []

    def body(rank):
        try:
            _rank_body(rank, 2, dist.ThreadComm(shared, rank), scene_name, steps, out, 0)
        except BaseException as e:               # noqa: BLE001  (a dead rank must not leave its peer in the barrier)
            errs.append(e)
            shared.barrier.abort()
    ts = [threading.Thread(target=body, args=(r,)) for r in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join(timeout=300)
    assert not errs, errs
    return sorted(out, key=lambda r: r["rank"])


def _check_stacks(E, res):
    r0, r1 = res
    assert r0["first_hit"] == r1["first_hit"] and r0["first_hit"] is not None and r0["first_hit"] > 0
    assert (r0["migrated_in"], r0["migrated_out"], r1["migrated_in"], r1["migrated_out"]) == (3, 0, 0, 3)
    assert r0["dynamic"] == 6 and r1["dynamic"] == 0 and r0["err"] == r1["err"] == 0 and not r1["pairs"]
    scene = E.scenes.approaching_stacks(height=3, gap=0.6, speed=3.0)
    ref = E.scenes.build_world(scene)
    ref.step(60)
    want = ref.download_state()["pos"][:6]
    ent, pos = np.asarray(r0["entities"]), np.asarray(r0["pos"], f32)
    got = np.zeros((6, 3), f32)
    # rank 0 holds: its own three boxes, the plane, and the three arrivals (entities 3..5 in appended slots)
    for e in range(6):
        slot = np.where(ent == e)[0][-1]
        got[e] = pos[slot]
    # body ids (hence pair and Gauss-Seidel order) differ after the move: solver-tolerance agreement, not bitwise
    assert np.abs(got - want).max() < 5e-3, np.abs(got - want).max()


def _check_chains(E, res):
    r0, r1 = res
    scene = _chains_scene(E)
    n = scene["dynamic"]
    assert r0["err"] == r1["err"] == 0
    assert r1["migrated_out"] > 0 and r1["migrated_out"] % 4 == 0, "whole chains move"
    assert r0["migrated_in"] == r1["migrated_out"] and r0["migrated_out"] == 0
    assert r0["dynamic"] + r1["dynamic"] == n
    assert r0["joints"] + r1["joints"] == len(scene["hinges"]["a"]), "every joint is solved on exactly one rank"
    # collision_exclusion travelled with the chains: no manifold between adjacent links anywhere
    for r in res:
        for a, b in r["pairs"]:
            if a < n and b < n:
                assert not (a // 4 == b // 4 and abs(a - b) == 1), (a, b)
    # moved chains keep moving on their new owner and nothing fell through the plane
    for r in res:
        pos = np.asarray(r["pos"], f32)
        assert pos[:, 1].min() > -0.05


def test_handover_between_two_ranks_on_one_device(gpu, E):
    _check_stacks(E, _run_threads("stacks", 60))


def test_chain_handover_carries_joints_and_exclusions(gpu, E):
    _check_chains(E, _run_threads("chains", 80))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _nccl_worker(rank, N, port, scene_name, steps, q):
    import traceback
    import torch
    import torch.distributed as dist_mod
    from edyn_b200 import dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist_mod.init_process_group("nccl", rank=rank, world_size=N, device_id=torch.device("cuda", rank))
    try:
        out = []
        _rank_body(rank, N, dist.TorchComm(dist_mod, rank, N), scene_name, steps, out, rank)
        q.put(out[0])
    except Exception:
        q.put(dict(rank=rank, error=traceback.format_exc()))
        os._exit(1)
    finally:
        dist_mod.destroy_process_group()


@pytest.mark.parametrize("scene_name,steps", [("stacks", 60), ("chains", 80)])
def test_handover_two_gpus_nccl(gpu, E, scene_name, steps):
    """The same hand-over with one process per GPU and the blobs travelling as device buffers over NCCL send / recv."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs; the threaded flavour above covers the library path on one")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, scene_name, steps, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    try:
        for _ in procs:
            r = q.get(timeout=180)
            assert "error" not in r, r["error"]
            res.append(r)
    finally:
        for p in procs:
            p.join(timeout=20)
            if p.is_alive():
                p.kill()
    res.sort(key=lambda r: r["rank"])
    (_check_stacks if scene_name == "stacks" else _check_chains)(E, res)
