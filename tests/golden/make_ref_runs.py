"""Regenerates tests/golden/ref_runs.npz: what the reference's OWN stepper_sequential (oracle/_ref/libedyn_stepper.so,
see make_whole_step.py) produced in the tests that compare against it, so that those tests run without the library.

    python tests/golden/make_ref_runs.py            # needs the reference at build time; the .npz travels, the reference does not

Contents:
  * free-running end states (no row order replayed): hinge_chains(8, 8) after 1000 steps
    (tests/test_zz_gpu_stepper_b2d.py), hinge_chains(4, 4) after 60 and 300 steps and hello_world after 24
    (tests/emu/lockstep.py vsref);
  * make_rigidbody's inverse inertia of 600 random bodies and the state after one step
    (tests/test_ref_stepper.py::test_python_make_rigidbody_mirror_matches_real_make_rigidbody);
  * for each scene of make_whole_step.SCENES, one 64-bit digest per step of the first LOCKSTEP_STEPS steps (state, AABBs,
    manifold set, point counts, island partition: step_digest) and the inverse inertia make_rigidbody derived
    (tests/test_ref_stepper.py::test_oracle_lockstep_with_real_stepper; the row order comes from whole_step.npz)."""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests.golden import make_whole_step as G  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_runs.npz")
LOCKSTEP_STEPS = 90
FREE_RUNS = {                       # name -> (edyn_b200.scenes factory, args, steps at which the state is kept)
    "chains_8x8": ("hinge_chains", (8, 8), (1000,)),
    "chains_4x4": ("hinge_chains", (4, 4), (60, 300)),
    "hello_world": ("hello_world", (), (24,)),
}


def pair_keys(p):
    p = np.asarray(p, np.uint64).reshape(-1, 2)
    return (p[:, 0] << np.uint64(32)) | p[:, 1]


def canonical_partition(labels):
    """Island labels renumbered in order of first appearance: equal arrays <=> equal partitions."""
    _, first, inv = np.unique(np.asarray(labels, np.int64), return_index=True, return_inverse=True)
    return np.argsort(np.argsort(first))[inv].astype(np.int64)


def step_digest(state, contacts, islands):
    """Digest of everything the lock-step tests compare bit for bit after a step."""
    h = hashlib.blake2b(digest_size=8)
    for k in ("pos", "orn", "linvel", "angvel", "aabb"):
        h.update(np.ascontiguousarray(state[k], np.float32).tobytes())
    keys = pair_keys(contacts["pairs"])
    order = np.argsort(keys, kind="stable")
    h.update(keys[order].tobytes())
    h.update(np.asarray(contacts["num"], np.uint32)[order].tobytes())
    h.update(canonical_partition(islands).tobytes())
    return np.frombuffer(h.digest(), np.uint64)[0]


def random_bodies(E):
    """The 600 bodies of the make_rigidbody mirror test: masses with 1 / (1 / m) == m in float (the harness hands the
    reference 1 / inv_mass)."""
    R = E.rigidbody
    rng, f = np.random.default_rng(7), np.float32
    defs = []
    while len(defs) < 600:
        m = f(rng.uniform(0.05, 50))
        if f(1) / (f(1) / m) != m:
            continue
        shape = [R.sphere_shape(float(rng.uniform(0.05, 2))), R.box_shape(tuple(rng.uniform(0.05, 2, 3))),
                 R.capsule_shape(float(rng.uniform(0.05, 1)), float(rng.uniform(0.05, 2)), int(rng.integers(3)))][rng.integers(3)]
        defs.append(R.RigidBodyDef(position=(10.0 * len(defs), 5, 0), mass=float(m), shape=shape))
    return R.bodies_soa(defs)


def main():
    import edyn_b200 as E
    from oracle import oracle as O
    O.build()
    assert O.ref_stepper() is not None, "oracle/_ref/libedyn_stepper.so missing: make -C oracle stepper"
    out = {}
    for name, (fn, a, marks) in FREE_RUNS.items():
        scene = getattr(E.scenes, fn)(*a)
        st = scene["settings"]
        r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
        G.populate(r, scene)
        n, done = scene["dynamic"], 0
        for m in marks:
            r.step(m - done)
            done = m
            x = r.state()
            out[f"{name}.{m}.pos"], out[f"{name}.{m}.linvel"] = x["pos"][:n], x["linvel"][:n]

    soa = random_bodies(E)
    r = O.RefWorld()
    r.add_bodies(soa)
    out["make_rigidbody.inertia_inv"] = r.inertia_inv()
    r.step(1)
    x = r.state()
    out["make_rigidbody.pos"], out["make_rigidbody.aabb"] = x["pos"], x["aabb"]

    for name in G.SCENES:
        scene = G.build_scene(E, name)
        st = scene["settings"]
        r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"])
        G.populate(r, scene)
        digests = []
        for _ in range(LOCKSTEP_STEPS):
            r.step(1)
            digests.append(step_digest(r.state(), r.contacts(), r.islands()))
        out[f"{name}.digests"] = np.asarray(digests, np.uint64)
        out[f"{name}.inertia_inv"] = r.inertia_inv()
        print(f"{name}: {LOCKSTEP_STEPS} steps, {int(r.contacts()['num'].sum())} points at the end")
    np.savez_compressed(OUT, **out)


if __name__ == "__main__":
    main()
