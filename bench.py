#!/usr/bin/env python
"""bench.py -- body-steps/sec of the Edyn per-step hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b2d|reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one fixed simulation step (broadphase -> narrowphase -> islands -> solve -> integrate) of the whole scene.

Workload (same at every N, so the driver's 1 -> 8 comparison is a STRONG-scaling one): BASELINE.json's config 5,
`chains_1048576` = 262 144 four-link hinge chains (1 048 576 bodies) resting on a plane -- the config the >= 6x
1 -> 8 target is quoted on.
  N = 1   the whole scene on one GPU.  The same line carries `workloads`: the other BASELINE configs at 1 GPU
          (`mixed_262144` -- the config the >= 10x CPU / >= 40 % roofline targets are quoted on --, `boxes_4096`,
          `spheres_65536`), each with its own value / e2e / roofline / cpu_baseline.
  N > 1   ONE scene, islands partitioned over the ranks (edyn_b200.dist.DeviceShardedWorld): every step each rank steps
          its islands, reduces the box of its bodies on the device, all-gathers the N boxes over NCCL (24 B per rank) and
          tests them; boxes within the broadphase margin trigger the island hand-over (device blobs over NCCL send/recv).
          One hand-over is forced inside the timed region: after the first timed step every rank r > 0 shoves its first
          column of chains into rank r-1's territory; `config.handover` reports what moved.

Keys beyond the base contract:
  roofline      velocity-solve kernel: algorithmic bytes (388 B per contact point per velocity iteration, 544 B per hinge
                per iteration, + 0.75 pass for the warm start; SURVEY.md section 8d) / mean CUDA-event duration of that
                kernel over the timed steps, against MEASURED_PEAKS.json's HBM copy bandwidth.
  cpu_baseline  rank 0, N = 1 only.  kind "reference": the reference's OWN stepper (oracle/_ref/libedyn_stepper.so =
                /root/reference/src/edyn compiled unmodified against oracle/entt_lite), execution_mode
                sequential_multithreaded on all host threads, on a bounded SLICE of the workload (same generator, fewer
                chains / a smaller pile: REF_SLICE) -- the full chain scene cannot be run by the reference in bounded
                time (entity_graph::insert_edge walks the plane's adjacency list for every new contact: quadratic in the
                bodies touching one static body).  `cpu_port` next to it: the oracle port (oracle/liboracle.so) on the
                FULL workload from the device's settled state, all threads -- the faster of the two CPU paths.
                Where the stepper library is absent the port is the cpu_baseline (kind "port").
  e2e           same metric through the C ABI with HOST buffers: every step uploads the body state from pinned
                host memory (b2d_upload_state), steps, and downloads it again (b2d_download_state).
--impl reference times the reference's CPU path: the real stepper on the slice above when oracle/_ref holds it (the line
also carries `port`, the oracle port on the full workload), else the oracle port on the full workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SETTLE_STEPS = 150            # untimed: lets the dropped bodies come to rest so contact counts are stationary
BYTES_PER_POINT_ITER = 388    # SURVEY.md section 8d
BYTES_PER_HINGE_ITER = 544
BYTES_PER_BODY_INTEGRATE = 276
DEFAULT_WORKLOAD = "chains_1048576"
OTHER_WORKLOADS = ["mixed_262144", "boxes_4096", "spheres_65536"]
# manifold capacity per body (max_manifolds is the user's reservation, like the reference's pool capacities): the measured
# high-water marks (AABB-overlap pairs incl. those without points: 6.92 / 4.6 / 5.4 / 1.0 per body) + 10-25 % head-room;
# an overflow raises ERR_MANIFOLD_CAPACITY and aborts the run
MANIFOLDS_PER_BODY = {"mixed_262144": 7.7, "boxes_4096": 6.0, "spheres_65536": 6.0, "chains_1048576": 1.25}


def make_scene(name, scale=1.0):
    import edyn_b200 as E
    if name == "mixed_262144":
        side = max(4, int(round(64 * scale ** (1 / 3))))
        return E.scenes.mixed_pile(side)
    if name == "boxes_4096":
        return E.scenes.boxes_on_plane(max(2, int(round(16 * scale ** (1 / 3)))))
    if name == "spheres_65536":
        return E.scenes.spheres_in_box(max(2, int(round(64 * scale ** 0.5))), 16, max(2, int(round(64 * scale ** 0.5))))
    if name == "chains_1048576":
        k = max(2, int(round(512 * scale ** 0.5)))
        return E.scenes.hinge_chains(k, k)
    raise SystemExit(f"unknown workload {name}")


def capacity(name, n_bodies):
    return max(4096, int(MANIFOLDS_PER_BODY.get(name, 10.0) * n_bodies))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.t = index, [], False, None

    def _nvml(self):
        """In-process NVML handle of CUDA device `index` (by UUID, so CUDA_VISIBLE_DEVICES cannot misalign them), or None."""
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                import torch
                uuid = "GPU-" + str(torch.cuda.get_device_properties(self.index).uuid)
                return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
            except Exception:
                return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            return None

    def _run(self):
        # NVML in process: a sample every 2 ms, so that a timed region of a few tens of milliseconds is covered by many
        # samples; nvidia-smi (one process launch per sample, ~100 ms) only where NVML cannot be loaded
        nv = self._nvml()
        if nv is not None:
            pynvml, h = nv
            try:
                mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
                bits = [pynvml.nvmlClocksThrottleReasonHwSlowdown, pynvml.nvmlClocksThrottleReasonHwThermalSlowdown,
                        pynvml.nvmlClocksThrottleReasonSwThermalSlowdown, pynvml.nvmlClocksThrottleReasonSwPowerCap]
                while not self.stop_flag:
                    sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                    why = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    self.rows.append([str(int(sm)), str(int(mx))] + ["Active" if why & b else "Not Active" for b in bits])
                    time.sleep(0.002)
                return
            except Exception:
                pass                                    # fall through to nvidia-smi with whatever was sampled so far
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def start(self):
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def stop(self):
        self.stop_flag = True
        if self.t:
            self.t.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def make_oracle(scene, threads):
    from oracle import oracle as O
    o = O.OracleWorld(vel_iters=scene["settings"]["velocity_iterations"], pos_iters=scene["settings"]["position_iterations"], threads=threads)
    o.add_bodies(scene["bodies"])
    if scene["hinges"]:
        h = scene["hinges"]
        o.add_hinges(h["a"], h["b"], h["pivot_a"], h["pivot_b"], h["axis_a"], h["axis_b"])
    if scene["exclusions"] is not None:
        o.add_exclusions(*scene["exclusions"])
    return o


def oracle_from_device(scene, w, threads):
    """Oracle world holding the device's current (settled) state, contacts included."""
    o = make_oracle(scene, threads)
    st = w.download_state(aabb=False)
    o.set_state(st["pos"], st["orn"], st["linvel"], st["angvel"])
    c = w.contacts()
    o.set_contacts(c["pairs"], c["num"], c["pts"], c["att"], c["lifetime"])
    return o


# ---------------------------------------------------------------------------------------------------------- CPU arm

# fraction of the workload's bodies the REAL reference stepper is timed on (it is 10-30x slower per body than the port and
# has a quadratic contact-creation step on scenes where everything touches one plane); throughput is per body-step
REF_SLICE = {"chains_1048576": 1.0 / 16, "mixed_262144": 1.0 / 8, "spheres_65536": 1.0, "boxes_4096": 1.0}


def have_real_reference():
    from oracle import oracle as O
    return O.ref_stepper() is not None


def make_ref_world(scene, threads):
    from oracle import oracle as O
    st = scene["settings"]
    r = O.RefWorld(vel_iters=st["velocity_iterations"], pos_iters=st["position_iterations"], threads=threads)
    r.add_bodies(scene["bodies"])
    if scene["hinges"]:
        h = scene["hinges"]
        r.add_hinges(h["a"], h["b"], h["pivot_a"], h["pivot_b"], h["axis_a"], h["axis_b"])
    if scene["exclusions"] is not None:
        r.add_exclusions(*scene["exclusions"])
    return r


def reference_real_isolated(args, name, steps, warmup, settle, budget_s):
    """reference_real in a child process: a fault inside the reference library (or a hang: the child is given the budget
    plus a margin) costs this leg, not the bench line.  Returns reference_real's tuple without the scene, or None."""
    cmd = [sys.executable, os.path.abspath(__file__), "--ref-child", json.dumps([name, steps, warmup, settle, budget_s, args.scale])]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=2.0 * budget_s + 120.0)
        if out.returncode != 0:
            raise RuntimeError(f"exit code {out.returncode}: {out.stderr[-300:]}")
        d = json.loads(out.stdout.strip().splitlines()[-1])
        return d["scene"], d["dynamic"], d["value"], d["dt"], d["sample"], d["cores"]
    except Exception as e:          # noqa: BLE001 -- whatever happened, the port still gives a CPU number
        print(f"bench: real reference stepper leg failed ({e}); reporting the port only", file=sys.stderr, flush=True)
        return None


def ref_child(spec):
    name, steps, warmup, settle, budget_s, scale = json.loads(spec)
    args = argparse.Namespace(scale=scale)
    scene, value, dt, sample, cores = reference_real(args, name, int(steps), int(warmup), int(settle), float(budget_s))
    print(json.dumps({"scene": scene["name"], "dynamic": scene["dynamic"], "value": value, "dt": dt, "sample": sample, "cores": cores}), flush=True)


def reference_real(args, name, steps, warmup, settle, budget_s):
    """The reference's own stepper_sequential (sequential_multithreaded, all host threads) on a slice of workload `name`.
    Settles as far as the time budget allows (the line says how far), then times `steps` steps."""
    cores = os.cpu_count() or 1
    scene = make_scene(name, args.scale * REF_SLICE.get(name, 1.0))
    threads, calib = cores, ""
    if cores > 16:
        # "all the host threads it can use": on a many-core host the reference's per-island tasks and parallel_for may run
        # better on fewer workers than hardware threads -- try both on a quarter-size scene and keep the faster
        small = make_scene(name, args.scale * REF_SLICE.get(name, 1.0) / 4)
        rates = {}
        for t in (cores, 16):
            w = make_ref_world(small, t)
            w.step(12)
            t0 = time.perf_counter()
            w.step(6)
            rates[t] = 6.0 / (time.perf_counter() - t0)
            del w
        threads = max(rates, key=rates.get)
        calib = f" (calibrated: {cores} workers {rates[cores]:.1f} steps/s, 16 workers {rates[16]:.1f} steps/s on {small['name']})"
    r = make_ref_world(scene, threads)
    t_start = time.perf_counter()
    n_settle, took = 0, []
    while n_settle < settle:
        t0 = time.perf_counter()
        r.step(1)
        took.append(time.perf_counter() - t0)
        n_settle += 1
        est = min(took[-2:])                                    # the step that creates all the contacts is an outlier
        if time.perf_counter() - t_start + 1.5 * est * (warmup + steps + 1) > budget_s:
            break
    r.step(warmup)
    t0 = time.perf_counter()
    r.step(steps)
    dt = time.perf_counter() - t0
    value = scene["dynamic"] * steps / dt
    sample = f"{scene['name']}: {scene['dynamic']} of the workload's dynamic bodies (same generator and settings), the reference's own " \
             f"stepper_sequential compiled from /root/reference against oracle/entt_lite, execution_mode sequential_multithreaded with " \
             f"{threads} workers{calib}, {n_settle} untimed settle steps, {steps} timed steps"
    return scene, value, dt, sample, threads

def reference_one(args, name, steps, warmup, settle, budget_s):
    """The CPU path (oracle port, all host threads) on the full workload `name`.  If the untimed settle would blow the
    time budget the settled state is approached with fewer settle steps and the line says so."""
    cores = os.cpu_count() or 1
    scene = make_scene(name, args.scale)
    o = make_oracle(scene, cores)
    t0 = time.perf_counter()
    o.step(1)
    per_step = time.perf_counter() - t0
    # keep the whole run inside the budget: settle as far as the budget allows (the dropped scenes are at rest long
    # before 150 steps; chains start 5 cm above the plane)
    n_settle = int(max(10, min(settle, (budget_s - per_step * (warmup + steps)) / max(per_step, 1e-6) - 1)))
    o.step(n_settle)
    for _ in range(warmup):
        o.step(1)
    t0 = time.perf_counter()
    o.step(steps)
    dt = time.perf_counter() - t0
    value = scene["dynamic"] * steps / dt
    sample = f"{scene['name']}: all {scene['dynamic']} dynamic bodies, same generator and settings as the device arm, " \
             f"{1 + n_settle} untimed settle steps, {steps} timed steps, {cores} threads (broadphase queries, narrowphase, per-island solve)"
    return scene, value, dt, sample, cores


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    port = None
    real = reference_real_isolated(args, args.workload, args.steps, args.warmup, args.ref_settle, args.ref_budget / 2) if have_real_reference() else None
    if real:
        kind = "reference"
        scene_name, n_dyn, value, dt, sample, cores = real
        _, pv, pdt, psample, pcores = reference_one(args, args.workload, min(args.steps, 10), min(args.warmup, 3), args.ref_settle, args.ref_budget / 2)
        port = {"value": pv, "unit": "body-steps/s", "cores": pcores, "kind": "port", "sample": psample}
    else:
        kind = "port"
        scene, value, dt, sample, cores = reference_one(args, args.workload, args.steps, args.warmup, args.ref_settle, args.ref_budget)
        scene_name, n_dyn = scene["name"], scene["dynamic"]
    line = {"impl": "reference", "metric": "body-steps/sec", "value": value, "unit": "body-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload if args.scale == 1.0 else f"{args.workload} x{args.scale}", "scene": scene_name,
                       "dynamic_bodies": n_dyn, "sample": sample},
            "cpu_baseline": {"value": value, "unit": "body-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "body-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    if port:
        line["port"] = port
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------- device arm

def solver_roofline(st, scene, step_ms):
    peak, peak_src = peaks()
    iters = scene["settings"]["velocity_iterations"]
    algo_bytes = (iters + 0.75) * (BYTES_PER_POINT_ITER * st["contact_points"] + BYTES_PER_HINGE_ITER * st["hinges"])
    achieved = algo_bytes / (st["solve_ms"] * 1e-3) / 1e9 if st["solve_ms"] > 0 else 0.0
    n_dyn = scene["dynamic"]
    integ_gbs = BYTES_PER_BODY_INTEGRATE * n_dyn / (st["integrate_ms"] * 1e-3) / 1e9 if st["integrate_ms"] > 0 else 0.0
    return {"bound": "hbm", "kernel": "velocity solve: k_island_tiles (small islands on chip; the launch also holds their integration and position iterations, "
                                      "so the fraction is understated where they dominate) + k_solve_df (ticket dataflow)", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes,
            "kernel_ms": st["solve_ms"], "kernel_share_of_step": st["solve_ms"] / step_ms if step_ms > 0 else None,
            "integrate": {"kernel": "k_integrate", "achieved": integ_gbs, "frac": integ_gbs / peak, "kernel_ms": st["integrate_ms"]}}


def traffic_for(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of the solve kernel per launch from the committed ncu capture."""
    for fn in ("traffic_r02.json", "traffic_r01.json"):
        p = os.path.join(ROOT, "profiles", fn)
        if os.path.exists(p):
            tj = json.load(open(p))
            ent = tj.get(name) if isinstance(tj.get(name), dict) else (tj if tj.get("workload") == name else None)
            if ent and "k_solve" in ent:
                return ent["k_solve"]["dram_bytes_read"] + ent["k_solve"]["dram_bytes_write"]
    return None


DUMP_MAX_BODIES = 1 << 18      # per workload: 13 floats a body, so the four workloads stay far below 64 MB


def dump_outputs(out_dir, name, state):
    """Writes the body state a caller of b2d_step receives (pos, orn, linvel, angvel) as out_dir/<workload>.<field>.npy,
    float32.  A workload with more bodies than DUMP_MAX_BODIES is sampled: the same seeded, sorted body indices every run."""
    n = len(state["pos"])
    idx = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_BODIES, replace=False)) if n > DUMP_MAX_BODIES else np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    for k in ("pos", "orn", "linvel", "angvel"):
        np.save(os.path.join(out_dir, f"{name}.{k}.npy"), np.ascontiguousarray(state[k][idx], np.float32))


def measure_single(args, name, local_rank, steps, warmup, cpu_seconds, sample_clocks, real_reference=False):
    """One workload, whole scene on one GPU: device-resident value, e2e through host buffers, roofline, CPU baseline."""
    import torch
    import edyn_b200 as E
    scene = make_scene(name, args.scale)
    n_dyn = scene["dynamic"]
    w = E.scenes.build_world(scene, device=local_rank, max_manifolds=capacity(name, len(scene["bodies"]["kind"])))
    w.step(SETTLE_STEPS)
    w.sync()
    stream = torch.cuda.ExternalStream(w.stream, device=local_rank)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local_rank) if sample_clocks else None
    if sampler:                                      # spans warm-up + timed region: 20 steps of a few ms are shorter than one nvidia-smi query
        sampler.start()
        for _ in range(30):
            w.step(1)
    for _ in range(warmup):
        w.step(1)
    w.sync()
    w.reset_timers()
    launches0 = w.stats()["kernel_launches"]
    e0.record(stream)
    for _ in range(steps):
        w.step(1)
    e1.record(stream)
    w.sync()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    st = w.stats()
    launches = st["kernel_launches"] - launches0 - 1        # minus the stats kernel itself
    value = n_dyn * steps / (ms * 1e-3)

    # ---- end to end through the C ABI with host buffers
    n_all = w.num_bodies
    pinned = {k: torch.empty((n_all, d), dtype=torch.float32).pin_memory() for k, d in (("pos", 3), ("orn", 4), ("linvel", 3), ("angvel", 3))}
    host = {k: v.numpy() for k, v in pinned.items()}
    w.download_state(aabb=False, out=host)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, name, host)
    e2e_steps = steps
    for _ in range(3):
        w.upload_state(host["pos"], host["orn"], host["linvel"], host["angvel"])
        w.step(1)
        w.download_state(aabb=False, out=host)
    w.sync()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(e2e_steps):
        w.upload_state(host["pos"], host["orn"], host["linvel"], host["angvel"])
        w.step(1)
        w.download_state(aabb=False, out=host)         # blocks until the step's results are on the host
    e1.record(stream)
    w.sync()
    wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max(e0.elapsed_time(e1), wall_ms)
    e2e_value = n_dyn * e2e_steps / (e2e_ms * 1e-3)
    bytes_state = n_all * 13 * 4

    roofline = solver_roofline(st, scene, ms / steps)
    roofline["traffic"] = traffic_for(name) if args.scale == 1.0 else None

    cpu = None
    if cpu_seconds > 0:
        cores = os.cpu_count() or 1
        o = oracle_from_device(scene, w, cores)
        o.step(1)                                   # untimed: first touch
        nsteps, t0 = 0, time.perf_counter()
        while nsteps < 3 or (time.perf_counter() - t0 < cpu_seconds and nsteps < 200):
            o.step(1)
            nsteps += 1
        dt = time.perf_counter() - t0
        cpu = {"value": n_dyn * nsteps / dt, "unit": "body-steps/s", "cores": cores, "kind": "port",
               "sample": f"{nsteps} steps of the same settled {scene['name']} state downloaded from the device "
                         f"(oracle/ CPU restatement of stepper_sequential; broadphase queries, narrowphase and per-island solve on {cores} threads)"}
    cpu_port = None
    if cpu and real_reference and have_real_reference():
        real = reference_real_isolated(args, name, 5, 2, min(args.ref_settle, 60), args.ref_real_seconds)
        if real:
            _, _, rv, _, rsample, rcores = real
            cpu_port, cpu = cpu, {"value": rv, "unit": "body-steps/s", "cores": rcores, "kind": "reference", "sample": rsample}
    if st["error_flags"]:
        raise SystemExit(f"{name}: device error flags {st['error_flags']}")
    res = {"value": value, "unit": "body-steps/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup,
           "config": {"workload": name if args.scale == 1.0 else f"{name} x{args.scale}", "scene": scene["name"], "dynamic_bodies": n_dyn,
                      "velocity_iterations": scene["settings"]["velocity_iterations"], "position_iterations": scene["settings"]["position_iterations"],
                      "settle_steps": SETTLE_STEPS, "manifolds": st["manifolds"], "contact_points": st["contact_points"], "hinges": st["hinges"],
                      "contact_colors": st["contact_colors"], "islands": st["islands"],
                      "l2": "inputs change every step and the per-step working set (rows + manifolds + bodies) exceeds the 126 MB L2 for the "
                            "two large configs; no explicit flush"},
           "gpu_launches": int(launches),
           "e2e": {"value": e2e_value, "unit": "body-steps/s", "h2d_bytes_per_step": bytes_state, "d2h_bytes_per_step": bytes_state, "steps": e2e_steps},
           "roofline": roofline}
    if cpu:
        res["cpu_baseline"] = cpu
    if cpu_port:
        res["cpu_port"] = cpu_port
    if clocks:
        res["clocks"] = clocks
    w.close()
    return res


def run_single(args, local_rank):
    top = measure_single(args, args.workload, local_rank, args.steps, args.warmup, 0 if args.no_cpu else args.cpu_seconds, True, real_reference=True)
    line = {"metric": "body-steps/sec", "value": top["value"], "unit": "body-steps/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": top["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(top["config"], parallelism="1 GPU: whole scene in one device world"),
            "clocks": top.get("clocks"), "gpu_launches": top["gpu_launches"], "e2e": top["e2e"], "roofline": top["roofline"]}
    for k in ("cpu_baseline", "cpu_port"):
        if k in top:
            line[k] = top[k]
    if args.workload == DEFAULT_WORKLOAD and args.scale == 1.0 and not args.only:
        subs = {}
        for name in OTHER_WORKLOADS:
            subs[name] = measure_single(args, name, local_rank, args.steps, args.warmup, 0 if args.no_cpu else args.cpu_seconds / 2, False)
        line["workloads"] = subs
    print(json.dumps(line), flush=True)


def run_sharded(args, world_size, rank, local_rank):
    """N > 1: ONE scene, islands partitioned over the ranks, strong scaling."""
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")       # the hand-over kernels first run inside the timed region
    import torch
    import torch.distributed as dist
    import edyn_b200 as E
    from edyn_b200 import dist as D
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)

    def barrier():
        dist.barrier()
        torch.cuda.synchronize()

    scene = make_scene(args.workload, args.scale)
    n_total = scene["dynamic"]
    labels = D.device_islands(scene, device=local_rank)            # island_manager's connected components, computed on the device
    comm = D.TorchComm(dist, rank, world_size)
    n_all = len(scene["bodies"]["kind"])
    sw = D.DeviceShardedWorld(scene, rank, world_size, comm, device=local_rank, labels=labels, slack=2.0 / world_size, pipeline=not args.exact_exchange,
                              max_manifolds=capacity(args.workload, int(n_all * (1.0 / world_size + 2.0 / world_size))))
    w = sw.world
    owner = sw.owner
    sw.step(SETTLE_STEPS)
    w.sync()
    stream = sw.ext
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # the forced hand-over: rank r > 0 shoves its first column of islands (lowest x) towards rank r-1
    push_ids = np.zeros(0, np.uint32)
    if rank > 0 and sw.local["dynamic"] > 0:
        b = sw.local["bodies"]
        dyn = np.where(b["kind"] == 0)[0]
        x = b["pos"][dyn, 0]
        push_ids = dyn[x < x.min() + 2.5].astype(np.uint32)          # one column of chains spans 2.1 in x, columns are 3.5 apart
    push_v = np.zeros((len(push_ids), 3), np.float32)
    push_v[:, 0] = -6.0

    w.set_timing(False)                 # the whole step is ONE graph launch (the per-kernel event ring splits it in three)
    for _ in range(args.warmup):
        sw.step(1)
    barrier()
    w.sync()
    launches0 = w.stats()["kernel_launches"]
    bytes0 = comm.bytes_sent
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    step_ms = []
    t_prev = time.perf_counter()
    e0.record(stream)
    for k in range(args.steps):
        if k == 1 and len(push_ids):
            w.upload_bodies(push_ids, linvel=push_v)
        sw.step(1)
        t_now = time.perf_counter(); step_ms.append((t_now - t_prev) * 1e3); t_prev = t_now
    e1.record(stream)
    w.sync()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    st = w.stats()
    launches = st["kernel_launches"] - launches0 - 1
    last_step_device_ms = st["last_step_ms"]                    # the last b2d_step alone, between its own two events
    # solver kernel time for the roofline note: a few more steps with the per-kernel events on (outside the timed region)
    w.set_timing(True); w.reset_timers()
    sw.step(5, exchange=False)
    w.sync()
    st = dict(st, **{k: w.stats()[k] for k in ("solve_ms", "integrate_ms")})
    w.set_timing(False)
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = n_total * args.steps / (ms_max * 1e-3)
    moved = torch.tensor([sw.migrated_in, sw.migrated_out, sw.handover_rounds, sw.halo_checks, sw.dynamic, comm.bytes_sent - bytes0], dtype=torch.int64, device="cuda")
    allmoved = [torch.zeros_like(moved) for _ in range(world_size)]
    dist.all_gather(allmoved, moved)
    allmoved = torch.stack(allmoved).cpu().numpy()

    # ---- end to end: host buffers in and out every step on every rank
    n_loc = w.num_bodies
    pinned = {k: torch.empty((n_loc, d), dtype=torch.float32).pin_memory() for k, d in (("pos", 3), ("orn", 4), ("linvel", 3), ("angvel", 3))}
    host = {k: v.numpy() for k, v in pinned.items()}
    w.download_state(aabb=False, out=host)
    e2e_steps = args.steps
    for _ in range(3):
        w.upload_state(host["pos"], host["orn"], host["linvel"], host["angvel"])
        sw.step(1)
        w.download_state(aabb=False, out=host)
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(e2e_steps):
        w.upload_state(host["pos"], host["orn"], host["linvel"], host["angvel"])
        sw.step(1)
        w.download_state(aabb=False, out=host)
    e1.record(stream)
    w.sync()
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([max(e0.elapsed_time(e1), wall_ms), float(n_loc)], dtype=torch.float64, device="cuda")
    tm = t.clone(); dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ts = t.clone(); dist.all_reduce(ts, op=dist.ReduceOp.SUM)
    e2e_value = n_total * e2e_steps / (float(tm[0].item()) * 1e-3)
    bytes_state = int(ts[1].item()) * 13 * 4

    if st["error_flags"]:
        raise SystemExit(f"rank {rank}: device error flags {st['error_flags']}")
    print(f"[rank {rank}] hand-over rounds (ms): {sw.handover_phases}; host ms per timed step: {[round(x, 2) for x in step_ms]}", file=sys.stderr, flush=True)
    if rank == 0:
        local_scene = dict(scene, dynamic=sw.dynamic)
        roofline = solver_roofline(st, local_scene, ms / args.steps)
        roofline["note"] = "rank 0's velocity-solve kernel over rank 0's constraints"
        srt = sorted(step_ms)
        line = {"metric": "body-steps/sec", "value": value, "unit": "body-steps/s", "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": args.workload if args.scale == 1.0 else f"{args.workload} x{args.scale}", "scene": scene["name"],
                           "dynamic_bodies": n_total, "dynamic_bodies_rank0": int(sw.dynamic),
                           "velocity_iterations": scene["settings"]["velocity_iterations"], "position_iterations": scene["settings"]["position_iterations"],
                           "settle_steps": SETTLE_STEPS, "manifolds_rank0": st["manifolds"], "contact_points_rank0": st["contact_points"], "hinges_rank0": st["hinges"],
                           "islands_rank0": st["islands"],
                           "parallelism": f"ONE scene, islands (connected components computed on the device) partitioned over {world_size} GPUs by x-slabs of equal "
                                          "body count; per step: b2d_step (one CUDA graph) + device reduction of the rank box and the fastest body speed + NCCL "
                                          "all-gather of 32 B/rank (the limiting collective: latency-bound) + copy to pinned memory; " +
                                          ("the host reads the boxes before the next step starts; " if args.exact_exchange else
                                           "the host reads the boxes of step k while step k+1 runs and widens the test margin by one step of closing travel "
                                           "(4 v_max dt + 2 g dt^2), so a hand-over still lands before the broadphase that needs it; ") +
                                          "island hand-over as device blobs over NCCL send/recv when boxes come within the margin",
                           "handover": {"bodies_in_per_rank": allmoved[:, 0].tolist(), "bodies_out_per_rank": allmoved[:, 1].tolist(),
                                        "rounds_per_rank": allmoved[:, 2].tolist(), "halo_checks_per_rank": allmoved[:, 3].tolist(),
                                        "dynamic_bodies_per_rank_after": allmoved[:, 4].tolist(),
                                        "collective_payload_bytes_per_rank_timed_region": allmoved[:, 5].tolist(),
                                        "forced": "after timed step 1 every rank r > 0 gives its first column of chains -6 m/s in x (b2d_upload_bodies)",
                                        "rank0_host_ms_per_step": {"median": srt[len(srt) // 2], "max": srt[-1]}, "rank0_last_step_device_ms": last_step_device_ms,
                                        "rank0_handover_round_ms": sw.handover_ms, "rank0_handover_phases_ms": sw.handover_phases,
                                        "rank0_host_ms_each_step": [round(x, 3) for x in step_ms]},
                           "l2": "per-step working set per rank exceeds L2 at N <= 4 (rows + manifolds + bodies); inputs change every step; no explicit flush"},
                "clocks": clocks, "gpu_launches": int(launches),
                "e2e": {"value": e2e_value, "unit": "body-steps/s", "h2d_bytes_per_step": bytes_state, "d2h_bytes_per_step": bytes_state, "steps": e2e_steps},
                "roofline": roofline}
        print(json.dumps(line), flush=True)
    sw.close()
    dist.destroy_process_group()


def run_device(args):
    import torch  # noqa: F401
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world_size > 1:
        run_sharded(args, world_size, rank, local_rank)
    else:
        torch.cuda.set_device(local_rank)
        run_single(args, local_rank)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2d", choices=["b2d", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD)
    ap.add_argument("--only", action="store_true", help="N = 1: skip the `workloads` sub-results of the other BASELINE configs")
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (development only; invalid as a bench value)")
    ap.add_argument("--ref-settle", type=int, default=SETTLE_STEPS)
    ap.add_argument("--ref-budget", type=float, default=200.0, help="reference arm: seconds the untimed settle + timed steps may take")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--ref-real-seconds", type=float, default=75.0, help="device arm: budget of the real reference stepper's cpu_baseline leg")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--ref-child", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--exact-exchange", action="store_true", help="N > 1: read every step's rank boxes before the next step starts (no look-ahead margin)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="N = 1, device arm: after the timed steps write each workload's body state as DIR/<workload>.<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b2d" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b2d --gpus 1")
    if args.ref_child:
        ref_child(args.ref_child)
        return
    if args.impl == "reference":
        run_reference(args)
    else:
        run_device(args)


if __name__ == "__main__":
    main()
