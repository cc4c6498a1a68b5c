"""TEST INFRASTRUCTURE.  The library's CUDA kernels, executed by the CPU emulation (tests/emu), in lock step with the
oracle through the normal Python adapter and C ABI -- the same comparison tests/test_gpu_parity.py makes on a B200: ordered
pair lists identical, post-solve state within 1e-5 (here: identical, glibc's sinf / cosf on both sides) with the oracle
replaying the device's Gauss-Seidel order, manifolds and joint impulses re-synchronised every step.

    python tests/emu/lockstep.py fixed|narrow|wide FIRST LAST [--tiles 0|1] [--steps N] [--restitution] [--mutate]     -> one JSON line
Runs in its own process because B2D_LIB has to be set before edyn_b200 is imported."""
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def lockstep(E, O, scene, steps, restitution_solver=False):
    import numpy as np
    w = E.scenes.build_world(scene, flags=E.world.FLAG_RESTITUTION_SOLVER if restitution_solver else 0)
    st = scene["settings"]
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    if restitution_solver:
        o.set_restitution_iterations(8, 3)          # no graph order handed over: the oracle's defaults are the device's conventions
    o.add_bodies(scene["bodies"])
    if scene["hinges"]:
        h = scene["hinges"]
        o.add_hinges(h["a"], h["b"], h["pivot_a"], h["pivot_b"], h["axis_a"], h["axis_b"])
    if scene["exclusions"] is not None:
        o.add_exclusions(*scene["exclusions"])
    worst = 0.0
    for s in range(steps):
        w.step(1)
        hi, pr = w.solver_order()
        o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
        o.set_order(hi, pr)
        o.run_phases(O.PH_SOLVE)
        g, c = w.download_state(), o.state()
        if {tuple(p) for p in w.pairs().tolist()} != {tuple(p) for p in o.pairs().tolist()}:
            return dict(ok=False, step=s, why="ordered broadphase pair lists differ")
        if not np.array_equal(w.islands(), o.islands()):
            return dict(ok=False, step=s, why="island labels differ")
        err = max(float(np.abs(g[k] - c[k]).max()) for k in ("pos", "orn", "linvel", "angvel", "aabb"))
        worst = max(worst, err)
        if err > 1e-5:
            return dict(ok=False, step=s, why=f"state differs by {err:.3e}")
        o.set_state(g["pos"], g["orn"], g["linvel"], g["angvel"])
        gc = w.contacts()
        o.set_contacts(gc["pairs"], gc["num"], gc["pts"], gc["att"], gc["lifetime"])
        if scene["hinges"]:
            o.set_hinge_impulses(w.hinge_impulses())
    stats = w.stats()
    w.close()
    return dict(ok=stats["error_flags"] == 0, worst=worst, points=int(stats["contact_points"]), flags=int(stats["error_flags"]))


def lockstep_with_mutations(E, O, scene, steps, seed):
    """Same comparison while user code interferes every 13th step: b2d_remove_bodies, b2d_remove_exclusions, b2d_add_bodies,
    b2d_upload_bodies (a patched velocity)."""
    import numpy as np
    R = E.rigidbody
    rng = np.random.default_rng(seed)
    st = scene["settings"]
    nb = len(scene["bodies"]["kind"])
    w = E.scenes.build_world(scene, max_bodies=nb + 16)
    o = O.OracleWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
    o.add_bodies(scene["bodies"])
    if scene["hinges"]:
        h = scene["hinges"]
        o.add_hinges(h["a"], h["b"], h["pivot_a"], h["pivot_b"], h["axis_a"], h["axis_b"])
    if scene["exclusions"] is not None:
        o.add_exclusions(*scene["exclusions"])
    kind = np.asarray(scene["bodies"]["kind"]).copy()
    alive = np.ones(len(kind), bool)
    excluded = list(zip(*[x.tolist() for x in scene["exclusions"]])) if scene["exclusions"] is not None else []
    events = 0
    for s in range(steps):
        if s and s % 13 == 0:
            what, movable = rng.integers(4), np.where(alive & (kind == 0))[0]
            if what == 0 and len(movable) > 4:
                b = int(rng.choice(movable))
                w.remove_bodies([b]); o.remove_bodies([b]); alive[b] = False
            elif what == 1 and excluded:
                a, b = excluded.pop()
                if alive[a] and alive[b]:
                    w.remove_exclusions([a], [b]); o.remove_exclusions([a], [b])
            elif what == 3 and len(kind) < nb + 16:
                d = R.RigidBodyDef(position=tuple(rng.uniform([-1, 2, -1], [1, 4, 1])), mass=float(rng.choice([0.5, 1.0, 2.0])), linvel=tuple(rng.uniform(-2, 2, 3)),
                                   shape=[R.sphere_shape(0.3), R.box_shape((0.3, 0.2, 0.25)), R.capsule_shape(0.15, 0.3, 1)][rng.integers(3)])
                soa = R.bodies_soa([d])
                w.add_bodies(soa); o.add_bodies(soa)
                kind, alive = np.append(kind, 0), np.append(alive, True)
            else:
                b = int(rng.choice(movable))
                lv, av = rng.uniform(-3, 3, (1, 3)).astype(np.float32), rng.uniform(-3, 3, (1, 3)).astype(np.float32)
                w.upload_bodies([b], linvel=lv, angvel=av)
                x = o.state()
                x["linvel"][b], x["angvel"][b] = lv[0], av[0]
                o.set_state(x["pos"], x["orn"], x["linvel"], x["angvel"])
            events += 1
        w.step(1)
        hi, pr = w.solver_order()
        o.run_phases(O.PH_BROAD | O.PH_NARROW | O.PH_ISLANDS)
        o.set_order(hi, pr)
        o.run_phases(O.PH_SOLVE)
        g, c = w.download_state(), o.state()
        if {tuple(p) for p in w.pairs().tolist()} != {tuple(p) for p in o.pairs().tolist()}:
            return dict(ok=False, step=s, why="ordered broadphase pair lists differ")
        err = max(float(np.abs(g[k][alive] - c[k][alive]).max()) for k in ("pos", "orn", "linvel", "angvel"))
        if err > 1e-5:
            return dict(ok=False, step=s, why=f"state differs by {err:.3e}")
        o.set_state(g["pos"], g["orn"], g["linvel"], g["angvel"])
        gc = w.contacts()
        o.set_contacts(gc["pairs"], gc["num"], gc["pts"], gc["att"], gc["lifetime"])
        if scene["hinges"]:
            o.set_hinge_impulses(w.hinge_impulses())
    flags = int(w.stats()["error_flags"])
    w.close()
    return dict(ok=flags == 0, worst=0.0, points=events, flags=flags)


def free_run_against_real_stepper(E):
    """No oracle in between: the kernels (emulated) and the reference's real stepper (its states recorded by
    tests/golden/make_ref_runs.py), both free-running from the same scene.  Hinge chains are insensitive to the sweep order
    (tiny islands at rest), so the two must simply agree; hello_world must be identical while the box falls."""
    import numpy as np
    from tests.golden import make_ref_runs as R
    runs = np.load(R.OUT)
    out = []
    for name, key in (("chains_64", "chains_4x4"), ("hello_world", "hello_world")):
        fn, a, marks = R.FREE_RUNS[key]
        scene = getattr(E.scenes, fn)(*a)
        w = E.scenes.build_world(scene)
        n, done = scene["dynamic"], 0
        for m in marks:
            w.step(m - done); done = m
            g = w.download_state()
            c = {k: runs[f"{key}.{m}.{k}"] for k in ("pos", "linvel")}
            out.append(dict(scene=name, step=m, dpos=float(np.abs(g["pos"][:n] - c["pos"]).max()), dvel=float(np.abs(g["linvel"][:n] - c["linvel"]).max())))
        w.close()
    return out


def main():
    kind, first, last = sys.argv[1], int(sys.argv[2]), int(sys.argv[3])
    tiles = sys.argv[sys.argv.index("--tiles") + 1] if "--tiles" in sys.argv else "1"
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 100
    restitution = "--restitution" in sys.argv
    from tests.emu import build
    os.environ["B2D_LIB"] = build.build()
    os.environ["B2D_GRAPH"] = "0"
    os.environ["B2D_TILES"] = tiles
    import edyn_b200 as E
    from oracle import oracle as O
    from tests.test_ref_stepper import random_scene, random_scene_wide
    fixed = [lambda: E.scenes.hello_world(), lambda: E.scenes.boxes_on_plane(3), lambda: E.scenes.spheres_in_box(4, 6, 4),
             lambda: E.scenes.mixed_pile(5, jitter=0.01), lambda: E.scenes.hinge_chains(2, 2)]
    out, t0 = [], time.time()
    if kind == "vsref":
        print(json.dumps(dict(results=free_run_against_real_stepper(E), seconds=0.0)))
        return
    for i in range(first, last):
        scene = fixed[i]() if kind == "fixed" else (random_scene_wide if kind == "wide" else random_scene)(E, O, i)
        res = lockstep_with_mutations(E, O, scene, steps, i) if "--mutate" in sys.argv else lockstep(E, O, scene, steps, restitution)
        res["scene"] = scene["name"]
        out.append(res)
    print(json.dumps(dict(results=out, seconds=time.time() - t0)))


if __name__ == "__main__":
    main()
