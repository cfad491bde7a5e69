#!/usr/bin/env python
"""bench.py — solver + integrator constraint-iterations/s (BASELINE.json metric) on synthetic scenes.

    python bench.py --gpus N --steps K --warmup W            our arm (libbepucuda through the C ABI)
    python bench.py --impl reference --steps K --warmup W    reference arm: the CPU oracle (restatement of the reference; the C# reference
                                                             itself cannot be built here) on all host cores, AVX2 8-wide like Vector<float>
    N > 1: launched under torch.distributed.run, one rank per GPU. The path shards by independent islands (SURVEY.md §8e): every rank
    simulates its own pile, no data-path collective, weak scaling.

A "step" is one Simulation.Solve: substeps x (incremental contact update, kinematic prepass, WarmStart with embedded integration per batch,
velocity iterations x Solve per batch) + the final pose pass. Workload = BASELINE configs[1]: ShapePile-style pile, 100k bodies, 8 substeps x 2
velocity iterations. Prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DT = 1.0 / 60.0


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bodies", type=int, default=100_000)
    ap.add_argument("--substeps", type=int, default=8)
    ap.add_argument("--iterations", type=int, default=2)
    ap.add_argument("--scene", default="shape_pile", choices=["shape_pile", "ragdolls", "fallback_stress"])
    ap.add_argument("--mode", default="auto", choices=["auto", "graph", "stream"], help="auto = the execution mode that measured fastest for the scene (DESIGN.md §8)")
    ap.add_argument("--no-configs", action="store_true", help="skip the side block with the other BASELINE configs (C3 ragdolls x2, C5 fallback stress, 1 M-body pile 4 x 2)")
    ap.add_argument("--config-steps", type=int, default=20)
    ap.add_argument("--strict", action="store_true", help="use the -fmad=false build")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--large-bodies", type=int, default=1_000_000, help="body count of the large pile in the configs block (the scene size BASELINE.json's north_star targets); 0 = skip it")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the one-graph-over-N-GPUs block")
    ap.add_argument("--sharded-bodies", type=int, default=1_000_000, help="N > 1: body count of the pile whose single constraint graph is split over the N GPUs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last timed step computed (body poses, velocities, world inverse "
                    "inertias, accumulated impulses) as DIR/<name>.npy, so that two builds can be compared on identical inputs; rank 0 only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def make_scene(args, seed):
    from bepuphysics2_b200 import scenes

    if args.scene == "shape_pile":
        return scenes.shape_pile(args.bodies, seed=seed)
    if args.scene == "ragdolls":
        return scenes.ragdolls(max(1, args.bodies // 16), seed=seed, motor=getattr(args, "ragdoll_motor", "motor"))
    return scenes.fallback_stress(args.bodies, hubs=max(1, args.bodies // 1000), seed=seed)


DUMP_MAX_BODIES = 400_000  # 108 B per body in the dump
DUMP_MAX_IMPULSES = 4 << 20  # floats: with the bodies, under 64 MiB in all


def _sample(a, limit, seed):
    """`a` itself when it has at most `limit` rows, otherwise the same seeded subset of rows on every run (kept in order)."""
    if a.shape[0] <= limit:
        return a
    return a[np.sort(np.random.default_rng(seed).choice(a.shape[0], size=limit, replace=False))]


def solve_outputs(sim):
    """What a caller of Simulation.Solve reads back from `sim`'s host buffers: per body the pose, the velocity and the world inverse inertia (padding
    floats dropped), and the accumulated impulses of every constraint, flattened in (batch, type batch, constraint, row) order."""
    bodies = sim.bodies
    impulses = [tb.accumulated_impulses.transpose(0, 2, 1).reshape(-1, tb.impulse_rows)[:tb.constraint_count].ravel() for tb in sim.type_batches()]
    rows = _sample(np.arange(bodies.shape[0]), DUMP_MAX_BODIES, seed=1)
    return {"body_poses": bodies[rows][:, 0:7].copy(), "body_velocities": bodies[rows][:, np.r_[8:11, 12:15]].copy(),
            "body_world_inverse_inertias": bodies[rows][:, np.r_[16:23, 24:31]].copy(),
            "accumulated_impulses": _sample(np.concatenate(impulses) if impulses else np.zeros(0, dtype=np.float32), DUMP_MAX_IMPULSES, seed=2)}


def device_solve_outputs(ts, sim):
    """solve_outputs of the state the last bepucuda_solve left on the device. The host buffers are restored afterwards, so that later uploads
    from them send what they would have sent without the dump."""
    kept_bodies = sim.bodies.copy()
    type_batches = sim.type_batches()
    kept_impulses = [tb.accumulated_impulses.copy() for tb in type_batches]
    ts.download_bodies()
    ts.download_impulses()
    out = solve_outputs(sim)
    sim.bodies[:] = kept_bodies
    for tb, kept in zip(type_batches, kept_impulses):
        tb.accumulated_impulses[:] = kept
    return out


def write_outputs(directory, outputs):
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64)
        np.save(os.path.join(directory, name + ".npy"), a)


def build_sim(args, seed):
    import bepuphysics2_b200 as bp
    from bepuphysics2_b200 import scenes

    scene = make_scene(args, seed)
    sim = bp.Simulation(bundle_width=8, fallback_batch_threshold=64, substeps=args.substeps, velocity_iterations=args.iterations)
    scenes.build(scene, sim)
    return sim, scene["description"]


class ClockSampler:
    """SM clock + throttle (clocks event) reasons sampled DURING the timed region: NVML every 5 ms from a thread (nvidia_ml_py), falling back to
    `nvidia-smi -lms 100` (B200_PROFILING.md recipe) when NVML is unavailable."""

    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device_index):
        self.device_index = device_index
        self.samples = []  # (sm_mhz, sm_max_mhz, set(reasons))
        self.proc = None
        self.thread = None
        self.stop_flag = threading.Event()
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may remap indices: resolve through the PCI bus id of the torch device when possible
            handle = None
            try:
                import torch

                bus = torch.cuda.get_device_properties(device_index).pci_bus_id
                dom = torch.cuda.get_device_properties(device_index).pci_domain_id
                dev = torch.cuda.get_device_properties(device_index).pci_device_id
                handle = pynvml.nvmlDeviceGetHandleByPciBusId(("%08x:%02x:%02x.0" % (dom, bus, dev)).encode())
            except Exception:
                handle = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.nvml, self.handle = pynvml, handle
        except Exception:
            self.nvml = None

    def _nvml_loop(self):
        n = self.nvml
        reasons_fn = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(n, "nvmlDeviceGetCurrentClocksThrottleReasons")
        bits = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}
        smax = n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)
        while not self.stop_flag.is_set():
            try:
                sm = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                mask = reasons_fn(self.handle)
                self.samples.append((float(sm), float(smax), {k for k, b in bits.items() if mask & b}))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nvml is not None:
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device_index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                try:
                    self.samples.append((float(parts[0]), float(parts[1]), {n for n, v in zip(names, parts[3:7]) if v.lower().startswith("active")}))
                except ValueError:
                    pass

    def stop(self):
        self.stop_flag.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.thread:
            self.thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no clock samples"], "samples": 0}
        reasons = set()
        for s in self.samples:
            reasons |= s[2]
        return {"sm_mhz": float(np.median([s[0] for s in self.samples])), "sm_max_mhz": max(s[1] for s in self.samples), "reasons": sorted(reasons), "samples": len(self.samples),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def load_traffic(bodies, kernel):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this workload (profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    try:
        with open(path) as f:
            for row in json.load(f)["captures"]:
                if row["bodies"] == bodies and row["kernel"] == kernel:
                    return row
    except Exception:
        pass
    return None


AUTO_MODE = {"shape_pile": "graph", "ragdolls": "graph", "fallback_stress": "graph"}  # updated from measurements (profiles/r02_summary.md)


def resolve_mode(args):
    return AUTO_MODE.get(args.scene, "graph") if args.mode == "auto" else args.mode


def side_configs(args):
    """The other BASELINE.json configs, each as (key, argparse overrides). configs[1] (C2) is the headline and is measured by main()."""
    out = [("c3_ragdoll_tube_10k_1x4", dict(scene="ragdolls", bodies=160_000, substeps=1, iterations=4, ragdoll_motor="motor")),
           ("c3_ragdoll_tube_10k_servo_8x2", dict(scene="ragdolls", bodies=160_000, substeps=8, iterations=2, ragdoll_motor="servo")),
           ("c5_fallback_stress_50k_1x4", dict(scene="fallback_stress", bodies=50_000, substeps=1, iterations=4))]
    if args.large_bodies > 0:
        out.append(("c4_pile_%dk_4x2_one_gpu" % (args.large_bodies // 1000), dict(scene="shape_pile", bodies=args.large_bodies, substeps=4, iterations=2)))
        out.append(("pile_%dk_8x2_one_gpu" % (args.large_bodies // 1000), dict(scene="shape_pile", bodies=args.large_bodies, substeps=8, iterations=2)))
    return out


def measure_config(args, overrides, torch, bp, modes, flush, peak, steps, with_cpu):
    """Device-resident throughput of one configuration (N = 1): `steps` solves, L2 flushed before each, CUDA events on the context stream."""
    import copy

    cfg = copy.copy(args)
    for k, v in overrides.items():
        setattr(cfg, k, v)
    sim, description = build_sim(cfg, seed=5)
    mode_name = resolve_mode(cfg)
    ts = bp.CudaTimestepper(sim, device=torch.cuda.current_device(), strict_fp=args.strict, execution_mode=modes[mode_name])
    ts.describe()
    ms = []
    for i in range(3 + steps):
        flush.fill_(1)
        torch.cuda.synchronize()
        ts.solve_device_only(DT)
        if i >= 3:
            ms.append(ts.timings().solve_ms)
    t = ts.timings()
    ts.close()
    step_ms = float(np.mean(ms))
    out = {"workload": "%s: %s; %d substeps x %d velocity iterations" % (cfg.scene, description, cfg.substeps, cfg.iterations), "execution_mode": mode_name, "ms_per_step": step_ms,
           "steps": len(ms), "value": int(t.constraint_iterations) / (step_ms * 1e-3), "unit": "constraint-iterations/s", "constraints": int(t.constraint_count),
           "device_batches": int(t.device_batch_count), "kernel_launches_per_step": int(t.kernel_launches),
           "algorithmic_gbs_whole_step": int(t.algorithmic_bytes) / (step_ms * 1e-3) / 1e9}
    out["roofline_frac_whole_step"] = out["algorithmic_gbs_whole_step"] / peak
    if with_cpu:
        frames = 1 if cfg.bodies > 300_000 else 2
        cb = cpu_reference_run(cfg, steps=frames, warmup=0 if cfg.bodies > 300_000 else 1, threads=args.cpu_threads)
        out["cpu_baseline"] = {"value": cb["value"], "ms_per_step": cb["ms_per_step"], "cores": cb["cores"], "kind": "port", "sample": "%d frame(s) of this workload" % frames}
    return out


def measure_sharded(args, torch, dist, bp, rank, world, local_rank, flush):
    """One pile's constraint graph over all ranks. Device time per step = max over ranks of the CUDA-event time around each rank's solve."""
    from bepuphysics2_b200 import scenes, sharding

    bodies, substeps, iterations = args.sharded_bodies, 4, 2
    scene = scenes.shape_pile(bodies, seed=5)
    sim = bp.Simulation(bundle_width=8, substeps=substeps, velocity_iterations=iterations)
    scenes.build(scene, sim)
    solver = sharding.ShardedSolver(sim, rank, world, local_rank, strict_fp=args.strict)
    gathered = [None] * world
    dist.all_gather_object(gathered, solver.export_handles())
    solver.import_handles(gathered)
    solver.describe()
    solver.synchronize()
    dist.barrier()
    steps = max(3, min(args.steps, 10))

    def step():
        flush.fill_(1)
        torch.cuda.synchronize()
        dist.barrier()
        solver.solve(DT)
        return solver.timings().solve_ms

    for _ in range(3):
        step()
    ms = sum(step() for _ in range(steps)) / steps
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    mine = torch.tensor([float(sum(tb["count"] for tb in solver.shard))], dtype=torch.float64, device="cuda")
    dist.all_reduce(mine, op=dist.ReduceOp.SUM)
    shared = int(((solver.masks & (solver.masks - 1)) != 0).sum())
    solver.close()
    dist.barrier()
    out = {"workload": "shape_pile bodies=%d substeps=%d velocity_iterations=%d, one constraint graph" % (bodies, substeps, iterations), "n_gpus": world, "scaling": "strong",
           "constraints": int(sim.constraint_count), "constraints_uploaded_over_ranks": int(mine.item()), "bodies_shared_between_ranks": shared,
           "ms_per_step": t.item(), "value": sim.constraint_count * substeps * iterations / (t.item() * 1e-3), "unit": "constraint-iterations/s", "steps": steps,
           "timing": "CUDA events around each rank's solve, max over ranks; L2 flushed and ranks aligned (barrier) before every step"}
    if rank == 0:
        # the same pile on this GPU alone, same numerics, for the strong-scaling denominator
        ts = bp.CudaTimestepper(sim, device=local_rank, strict_fp=args.strict, execution_mode=bp.native.EXEC_GRAPH)
        ts.describe()
        ts.synchronize()

        def single():
            flush.fill_(1)
            torch.cuda.synchronize()
            ts.solve_device_only(DT)
            return ts.timings().solve_ms

        for _ in range(3):
            single()
        out["single_gpu_ms_per_step"] = sum(single() for _ in range(steps)) / steps
        ts.close()
    dist.barrier()
    return out


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def usable_cpu_count():
    """Threads we can really run: the scheduler affinity mask capped by the cgroup CPU quota (a 128-CPU box may grant a container far fewer)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) // int(period))))
    except Exception:
        pass
    return max(1, n)


def cpu_reference_run(args, steps, warmup, threads):
    """The oracle (CPU restatement of the reference solver, AVX2 8-wide lanes, OpenMP over bundles within each batch stage) on the same workload."""
    from oracle import binding as ob

    sim, desc = build_sim(args, seed=5)
    threads = threads or usable_cpu_count()
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")
    for _ in range(warmup):
        ob.solve(sim, DT, threads=threads, simd=True)
    t0 = time.perf_counter()
    for _ in range(steps):
        ob.solve(sim, DT, threads=threads, simd=True)
    dt = time.perf_counter() - t0
    ci_per_step = sim.constraint_count * args.substeps * args.iterations
    return {"value": ci_per_step * steps / dt, "ms_per_step": dt / steps * 1e3, "cores": threads, "constraints": sim.constraint_count, "description": desc, "sim": sim}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args, args.steps, args.warmup, args.cpu_threads)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, solve_outputs(r["sim"]))
    line = {
        "impl": "reference", "metric": "constraint-iterations/sec (solver+integrator)", "value": r["value"], "unit": "constraint-iterations/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, r["description"]),
        "cpu_baseline": {"value": r["value"], "unit": "constraint-iterations/s", "cores": r["cores"], "kind": "port",
                         "sample": "%d full frames of the same workload (C++ restatement of the reference solver, AVX2 8-wide, one worker per core with spin syncs between batch stages; the C# reference cannot be built here)" % args.steps},
        "e2e": {"value": r["value"], "unit": "constraint-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def workload_config(args, description):
    return {"workload": "%s: %s; %d substeps x %d velocity iterations, dt 1/60" % (args.scene, description, args.substeps, args.iterations),
            "bodies_per_gpu": args.bodies, "substeps": args.substeps, "velocity_iterations": args.iterations, "parallelism": "independent islands per GPU, no collective"}


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    import torch

    import bepuphysics2_b200 as bp
    from bepuphysics2_b200.native import EXEC_GRAPH, EXEC_STREAM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; libbepucuda has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        # stdout carries exactly one JSON line: NCCL_DEBUG=VERSION (set on the GPU boxes) prints a banner to stdout, WARN does not; other levels go to stderr
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    modes = {"graph": EXEC_GRAPH, "stream": EXEC_STREAM}
    args.mode = resolve_mode(args)
    mode = modes[args.mode]

    sim, description = build_sim(args, seed=5)  # every rank owns an independent island: the same pile on every rank, so ranks differ only by their GPU
    ts = bp.CudaTimestepper(sim, device=local_rank, strict_fp=args.strict, execution_mode=mode)
    ts.register_host_buffers()
    ts.describe()
    ts.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput: K solves, L2 flushed before each, timed with CUDA events on the context stream ----
    def solve_once_timed():
        flush.fill_(1)
        torch.cuda.synchronize()
        ts.solve_device_only(DT)
        return ts.timings().solve_ms  # get_timings synchronizes the context stream

    for _ in range(max(args.warmup, 3)):
        solve_once_timed()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    total_ms = 0.0
    for _ in range(args.steps):
        total_ms += solve_once_timed()
    barrier()
    clocks = sampler.stop()
    t = ts.timings()
    ci_per_step = int(t.constraint_iterations)
    launches_per_step = int(t.kernel_launches)
    alg_bytes_per_step = int(t.algorithmic_bytes)
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, device_solve_outputs(ts, sim))

    # ---- end to end through the C ABI with host buffers: H2D of bodies + prestep + impulses, solve, D2H of bodies + impulses ----
    for _ in range(2):
        ts.refresh()
        ts.solve(DT, download=True)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ts.refresh()
        ts.solve(DT, download=True)
    ts.synchronize()
    e2e_s = time.perf_counter() - t0
    te = ts.timings()
    h2d, d2h = int(te.h2d_bytes), int(te.d2h_bytes)

    # ---- end to end WITH a topology change every step (what a frame after collision detection looks like): the whole constraint description is
    # ---- re-uploaded (begin / upload_type_batch / end_constraints: transposition, ownership analysis, fallback levelisation, graph re-capture)
    topo = None
    if rank == 0:
        for _ in range(2):
            ts.describe()
            ts.solve(DT, download=True)
        ts.synchronize()
        topo_steps = max(3, min(args.steps, 6))
        t0 = time.perf_counter()
        for _ in range(topo_steps):
            ts.describe()
            ts.solve(DT, download=True)
        ts.synchronize()
        topo_s = time.perf_counter() - t0
        tt = ts.timings()
        topo = {"value": ci_per_step * topo_steps / topo_s, "unit": "constraint-iterations/s", "ms_per_step": topo_s / topo_steps * 1e3, "steps": topo_steps,
                "h2d_bytes_per_step": int(tt.h2d_bytes), "d2h_bytes_per_step": int(tt.d2h_bytes),
                "what": "every step: upload bodies + begin/upload/end_constraints (full topology rebuild) + solve + download bodies and impulses"}

    # ---- per-stage device time (event pair around every launch) for the roofline of the dominant kernel ----
    prof = None
    if rank == 0:
        flush.fill_(1)
        torch.cuda.synchronize()
        ts.profile_stages(DT)
        flush.fill_(1)
        torch.cuda.synchronize()
        prof = ts.profile_stages(DT).as_dict()

    # ---- end to end with the device-side contact update (SURVEY.md §8 f2): accumulated impulses stay on the device and are redistributed there from
    # ---- the old to the new feature ids; per step the host sends the motion half of the bodies, the new prestep data and the new feature ids, and
    # ---- reads back the motion half of the bodies only
    resident = None
    if args.scene == "shape_pile":  # every rank (its own island), like the full-refresh leg
        pool, _ = ts.contact_feature_pool(np.random.default_rng(11))  # one pinned block, like a BufferPool
        ts.register_array(pool)
        ts.describe()
        ts.set_contact_feature_pool(pool)
        for _ in range(2):
            ts.update_contacts_from_pool(pool)
            ts.solve_device_only(DT)
            ts.download_body_motion()
        ts.synchronize()
        barrier()
        r_steps = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(r_steps):
            ts.update_contacts_from_pool(pool)
            ts.solve_device_only(DT)
            ts.download_body_motion()
        ts.synchronize()
        r_s = time.perf_counter() - t0
        tr = ts.timings()
        resident = {"value": ci_per_step * r_steps / r_s, "unit": "constraint-iterations/s", "ms_per_step": r_s / r_steps * 1e3, "steps": r_steps,
                    "h2d_bytes_per_step": int(tr.h2d_bytes), "d2h_bytes_per_step": int(tr.d2h_bytes),
                    "what": "every step: upload the motion half of the bodies (64 B / body) + prestep + contact feature ids, redistribute the resident impulses on the device, solve, download the motion half of the bodies"}

    # ---- device-side batch colouring of this workload's constraint list (SURVEY.md §8 f3): bepucuda_color_constraints vs the host mirror's
    # ---- sequential Solver.Add batch search (C++, one thread), wall clock including the reference upload and the batch-index download
    def side_block(fn):
        """A side block never takes the headline line down with it: on failure its entry carries the error text instead."""
        try:
            return fn()
        except Exception as e:  # noqa: BLE001
            return {"error": "%s: %s" % (type(e).__name__, e)}

    def measure_colouring():
        from bepuphysics2_b200 import coloring

        scene_for_refs = make_scene(args, 5)
        refs = coloring.scene_references(scene_for_refs)
        colouring = {"constraints": int(refs.shape[0]), "what": "batch index per constraint, identical to sequential first fit in the stated order (tests/test_coloring.py)"}
        for order, name in ((1, "hashed_order"), (0, "insertion_order")):
            ts.color_constraints(refs, sim.body_count, 64, order=order)
            t0 = time.perf_counter()
            _, n_batches, rounds = ts.color_constraints(refs, sim.body_count, 64, order=order)
            colouring[name] = {"ms": (time.perf_counter() - t0) * 1e3, "batches": int(n_batches), "device_rounds": int(rounds)}
        from bepuphysics2_b200 import scenes as scenes_mod

        host_sim = bp.Simulation(bundle_width=8, fallback_batch_threshold=64, substeps=args.substeps, velocity_iterations=args.iterations)
        t0 = time.perf_counter()
        scenes_mod.build(scene_for_refs, host_sim)
        colouring["host_solver_add_ms"] = (time.perf_counter() - t0) * 1e3
        colouring["host_solver_add_what"] = "Bodies.Add + Solver.Add of every constraint in the C++ host mirror, one thread (batch search AND writing the type batches)"
        del host_sim
        return colouring

    colouring = side_block(measure_colouring) if rank == 0 and world == 1 and not args.no_configs else None

    # ---- PredictBoundingBoxes on the resident body state (SURVEY.md §8 f4): wall clock of the C-ABI call, i.e. activities up (8 B / body), the kernel,
    # ---- bounds + margins + activities down (40 B / body)
    def measure_predict():
        from bepuphysics2_b200 import native as native_mod

        rng = np.random.default_rng(3)
        nb = sim.body_count
        shapes = np.zeros(nb, dtype=native_mod.BODY_SHAPE_DTYPE)
        shapes["type"] = rng.choice([0, 1, 2, 4], size=nb)
        shapes["a"], shapes["b"], shapes["c"] = rng.uniform(0.3, 1.5, size=(3, nb)).astype(np.float32)
        shapes["maximum_speculative_margin"] = 3.40282347e+38
        shapes["allow_expansion_beyond_speculative_margin"] = 1
        activities = np.zeros(nb, dtype=native_mod.BODY_ACTIVITY_DTYPE)
        activities["sleep_threshold"], activities["minimum_timesteps_under_threshold"] = 0.01, 32
        ts.set_body_shapes(shapes)
        for _ in range(2):
            ts.predict_bounding_boxes(DT, activities)
        t0 = time.perf_counter()
        for _ in range(10):
            bounds = ts.predict_bounding_boxes(DT, activities)
        p_ms = (time.perf_counter() - t0) * 1e3 / 10
        predict = {"bodies": int(nb), "ms_per_call": p_ms, "bodies_per_s": nb / (p_ms * 1e-3), "valid_bounds": int((bounds[:, 7] == 1).sum()),
                   "what": "bepucuda_predict_bounding_boxes through the C ABI, pageable host buffers: 8 B / body up, 40 B / body down, one kernel (168 B / body of HBM traffic)"}
        return predict

    predict = side_block(measure_predict) if rank == 0 and world == 1 and not args.no_configs else None

    configs = None
    if rank == 0 and world == 1 and not args.no_configs and args.scene == "shape_pile":
        ts.close()
        ts = None
        peak_for_configs, _ = load_peaks()
        configs = {}
        for key, overrides in side_configs(args):
            configs[key] = side_block(lambda: measure_config(args, overrides, torch, bp, modes, flush, peak_for_configs, args.config_steps, with_cpu=not args.no_cpu_baseline))

    # ---- N > 1: ONE constraint graph over the N GPUs (SURVEY.md §8e), next to the N independent islands above: the 1M-body pile of configs[4],
    # ---- constraints split by body slab, shared body records pushed over NVLink by the stage kernels (bepucuda_shard_*); strong scaling
    sharded = None
    if dist is not None and not args.no_sharded and args.scene == "shape_pile":
        sharded = measure_sharded(args, torch, dist, bp, rank, world, local_rank, flush)

    per_rank_ms = [total_ms / args.steps]
    if dist is not None:
        gathered = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([total_ms / args.steps], dtype=torch.float64, device="cuda"))
        per_rank_ms = [float(g.item()) for g in gathered]
    times = torch.tensor([total_ms, e2e_s * 1e3, (resident["ms_per_step"] * resident["steps"]) if resident is not None else 0.0], dtype=torch.float64, device="cuda")
    counts = torch.tensor([float(ci_per_step)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
    total_ms_max, e2e_ms_max, resident_ms_max = times.tolist()
    if resident is not None:  # whole job: all ranks' constraint-iterations over the slowest rank's time
        resident["ms_per_step"] = resident_ms_max / resident["steps"]
        resident["value"] = counts.item() * resident["steps"] / (resident_ms_max * 1e-3)
    ci_all = counts.item()

    if rank == 0:
        peak, peak_source = load_peaks()
        value = ci_all * args.steps / (total_ms_max * 1e-3)
        e2e_value = ci_all * e2e_steps / (e2e_ms_max * 1e-3)
        roof_extra = {}
        # Dominant kernel: constraint_stage_kernel<Solve>. Its launches sit inside a CUDA graph with programmatic-dependent-launch edges, so its time
        # inside the timed region = (its share of the per-launch event-timed stage profile, taken right after the timed region on the same
        # stream) x (the event-timed step). The fully serialised event-per-launch figure is reported next to it.
        launches = prof["solve"]["launches"]
        share = prof["solve"]["ms"] / sum(v["ms"] for v in prof.values())
        roof_bytes, roof_ms = prof["solve"]["algorithmic_bytes"], share * total_ms / args.steps
        roof_kernel = "constraint_stage_kernel<Solve> (%d launches per step, %.0f%% of the step)" % (launches, 100 * share)
        roof_extra = {"share_of_step": share, "achieved_serialised_launches": prof["solve"]["algorithmic_bytes"] / (prof["solve"]["ms"] * 1e-3) / 1e9,
                      "whole_step_achieved": alg_bytes_per_step / (total_ms / args.steps * 1e-3) / 1e9}
        achieved = roof_bytes / (roof_ms * 1e-3) / 1e9
        traffic_row = load_traffic(args.bodies, "constraint_stage_kernel<Solve>") if args.scene == "shape_pile" else None
        traffic = None
        if traffic_row:
            traffic = traffic_row["dram_bytes_per_launch"]
            roof_extra["traffic_source"] = traffic_row["source"]
            roof_extra["traffic_launch"] = traffic_row["launch"]
            roof_extra["traffic_launch_algorithmic_bytes"] = traffic_row["algorithmic_bytes_per_launch"]
            roof_extra["mean_algorithmic_bytes_per_launch"] = roof_bytes / launches
        line = {
            "metric": "constraint-iterations/sec (solver+integrator)", "value": value, "unit": "constraint-iterations/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, description), execution_mode=args.mode, numerics="strict(-fmad=false)" if args.strict else "fast(fma)", l2="flushed (256 MiB write) before every timed step",
                           constraints_per_gpu=int(t.constraint_count), device_batches=int(t.device_batch_count), stages_per_step=int(t.stage_count)),
            "e2e": {"value": e2e_value, "unit": "constraint-iterations/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms_max / e2e_steps, "steps": e2e_steps,
                    "topology": "unchanged between steps (bodies + prestep + impulses re-uploaded, results downloaded)"},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": roof_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                         "peak_source": peak_source, "algorithmic_bytes_per_step": alg_bytes_per_step, **roof_extra},
            "stage_profile_ms": {k: round(v["ms"], 4) for k, v in (prof or {}).items()},
        }
        line["ms_per_step_per_rank"] = per_rank_ms
        if resident is not None:
            # Headline end-to-end figure = the frame a host with the device-side contact update (SURVEY.md §8 f2) runs: per step it uploads the motion
            # half of the bodies, the new prestep data and the new contact feature ids, and downloads the motion half of the bodies; accumulated
            # impulses never cross the bus. The full-refresh frame (everything up, everything down) stays next to it.
            line["e2e_full_refresh"] = line["e2e"]
            line["e2e"] = {"value": resident["value"], "unit": resident["unit"], "h2d_bytes_per_step": resident["h2d_bytes_per_step"], "d2h_bytes_per_step": resident["d2h_bytes_per_step"],
                           "ms_per_step": resident["ms_per_step"], "steps": resident["steps"],
                           "path": "bepucuda_upload_body_motion + bepucuda_update_contacts (prestep + feature ids; impulses resident, redistributed on the device) + bepucuda_solve + bepucuda_download_body_motion",
                           "topology": "unchanged between steps"}
        if topo is not None:
            line["e2e_topology_change"] = topo
        if resident is not None:
            line["e2e_resident_impulses"] = resident
        if colouring is not None:
            line["device_colouring"] = colouring
        if predict is not None:
            line["predict_bounding_boxes"] = predict
        if configs is not None:
            line["configs"] = configs
        if sharded is not None:
            line["one_graph_sharded"] = sharded
        if not args.no_cpu_baseline and world == 1:  # the CPU baseline is reported at N = 1 only
            cb = cpu_reference_run(args, steps=3, warmup=1, threads=args.cpu_threads)
            c1 = cpu_reference_run(args, steps=1, warmup=0, threads=1)  # the reference's own benchmarks run single-threaded (ShapePileBenchmark.cs:L228)
            line["cpu_baseline"] = {"value": cb["value"], "unit": "constraint-iterations/s", "cores": cb["cores"], "kind": "port",
                                    "sample": "3 full frames of the same workload after 1 warm-up (C++ restatement of the reference solver, AVX2 8-wide, one worker per core with spin syncs between batch stages; %.1f ms/frame)" % cb["ms_per_step"],
                                    "single_thread": {"value": c1["value"], "ms_per_step": c1["ms_per_step"], "sample": "1 frame, 1 thread, same code"}}
        print(json.dumps(line))
    if ts is not None:
        ts.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
