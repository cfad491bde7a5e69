"""PredictBoundingBoxes over every built-in shape type on the device (bepucuda_set_body_collidables path): one JSON line for a mixed world.

    python tests/tools/shape_bounds_timing.py [--bodies 100000] [--iters 50] [--out OUT.json]

World: `--bodies` bodies over a seeded library (64 of each primitive and of triangles, 64 hulls of 20-64 points at W = 8, 256 compounds and 64 big
compounds of 2-16 children, one mesh of 10 k and one of 1 M triangles, with a handful of mesh bodies); hulls and compounds are shared by many bodies.
Reports device time per class kernel (torch.profiler, CUDA activity, a run of its own), device time of the whole call (CUDA events on the context
stream, activity upload and bounds download included), wall clock through the C ABI, bodies/s, a compulsory-traffic model per class, the CPU oracle
on the same world for scale, and whether the device result is bit-identical to the oracle. The GPU's name and power limit are part of the record."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import bepuphysics2_b200 as bp  # noqa: E402
from bepuphysics2_b200 import scenes  # noqa: E402
from oracle import shape_bounds as osb  # noqa: E402

DT = 1.0 / 60.0
KERNELS = {"per_body": "shape_bounds_body_kernel", "hull": "shape_bounds_hull_kernel", "compound": "shape_bounds_compound_kernel",
           "mesh_chunks": "shape_bounds_mesh_chunk_kernel", "mesh_finish": "shape_bounds_mesh_finish_kernel"}


def traffic_model(world):
    """Bytes a pass has to move at least, per class: every body reads its motion (96 B: pose, velocity, local inertia), its 16-B collidable and 8-B
    activity and writes the activity and 32 B of bounds; hull / compound / mesh bodies read their motion and collidable again in their own kernel.
    Shape data shared by many bodies is counted once (it is read from L2 after the first body); each mesh body streams its triangles (36 B each)."""
    lib, c = world["library"], world["collidables"]["shape"]
    exists = (c >> 31) == 1
    types, index = (c >> 24) & 0x7F, c & 0xFFFFFF
    n = c.shape[0]
    hull_bodies = int((exists & (types == 5)).sum())
    compound_sel = exists & ((types == 6) | (types == 7))
    mesh_sel = exists & (types == 8)
    mesh_triangles = int(lib.meshes["triangle_count"][index[mesh_sel]].sum())
    return {
        "per_body": n * (96 + 16 + 8 + 8) + int((exists & (types <= 4)).sum()) * 32,
        "hull": hull_bodies * (96 + 16 + 32) + lib.hull_points.nbytes + lib.hulls.nbytes,
        "compound": int(compound_sel.sum()) * (96 + 16 + 32) + lib.compound_children.nbytes + lib.compounds.nbytes + lib.big_compounds.nbytes,
        "mesh": int(mesh_sel.sum()) * (96 + 16 + 32) + mesh_triangles * 36,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bodies", type=int, default=100_000)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement only runs on the GPU")
    rng = np.random.default_rng(2026)
    library = scenes.shape_library(rng, hull_width=8, primitives=64, hulls=64, hull_points=(20, 64), compounds=256, big_compounds=64, compound_children=(2, 16),
                                   mesh_triangle_counts=(10_000, 1_000_000))
    weights = {0: 1, 1: 1, 2: 1, 3: 1, 4: 1, 5: 2, 6: 2, 7: 0.5, 8: 4.0 / a.bodies * 19.0}  # about four mesh bodies
    world = scenes.shape_world(a.bodies, seed=7, library=library, type_weights=weights)
    integ = bp.IntegratorDesc.default()
    sim = bp.Simulation(integrator=integ)
    sim.add_bodies(world["bodies"])
    ts = bp.CudaTimestepper(sim, strict_fp=True)
    ts.describe()
    ts.set_shape_library(library)
    ts.set_body_collidables(world["collidables"])
    activities = world["activities"].copy()
    for _ in range(5):  # warm-up: module load, first-touch of every buffer
        ts.predict_bounding_boxes(DT, activities)

    wall, dev = [], []
    for _ in range(a.iters):
        ts.event_record(0)
        t = time.perf_counter()
        ts.predict_bounding_boxes(DT, activities)
        wall.append(time.perf_counter() - t)
        ts.event_record(1)
        ts.synchronize()
        dev.append(ts.event_elapsed_ms(0, 1))

    from torch.profiler import ProfilerActivity, profile

    per_kernel = {k: [] for k in KERNELS}
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            ts.predict_bounding_boxes(DT, activities)
    for ev in prof.events():
        for k, name in KERNELS.items():
            if name in ev.name and ev.device_type.name == "CUDA":
                per_kernel[k].append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
    kernel_ms = {k: (float(np.median(v)) / 1e3 if v else None) for k, v in per_kernel.items()}

    # parity of the timed world (a fresh pair of activity arrays), and the CPU oracle for scale
    want_act, got_act = world["activities"].copy(), world["activities"].copy()
    t = time.perf_counter()
    want = osb.predict_bounding_boxes_collidables(world["bodies"], world["collidables"], want_act, library, DT, integ)
    oracle_s = time.perf_counter() - t
    got = ts.predict_bounding_boxes(DT, got_act)
    identical = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)) and np.array_equal(got_act.view(np.uint8), want_act.view(np.uint8)))
    ts.close()

    types = (world["collidables"]["shape"] >> 24) & 0x7F
    exists = (world["collidables"]["shape"] >> 31) == 1
    model = traffic_model(world)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()
    result = {
        "what": "bepucuda_predict_bounding_boxes, set_body_collidables path, strict build",
        "gpu": gpu[0] if gpu else torch.cuda.get_device_name(0),
        "bodies": a.bodies,
        "bodies_per_type": {str(t): int((exists & (types == t)).sum()) for t in range(9)},
        "bodies_without_builtin_bounds": int((~exists | (types > 8)).sum()),
        "mesh_triangles_per_body": [int(x) for x in library.meshes["triangle_count"][(world["collidables"]["shape"] & 0xFFFFFF)[exists & (types == 8)]]],
        "iters": a.iters,
        "call_device_ms_median": float(np.median(dev)),
        "call_wall_ms_median": float(np.median(wall) * 1e3),
        "bodies_per_s_wall": float(a.bodies / np.median(wall)),
        "kernel_device_ms_median": kernel_ms,
        "traffic_model_bytes": model,
        "traffic_model_gb_per_s": {k: model[k] / (ms * 1e-3) / 1e9 for k, ms in (("per_body", kernel_ms["per_body"]), ("hull", kernel_ms["hull"]), ("compound", kernel_ms["compound"]),
                                   ("mesh", (kernel_ms["mesh_chunks"] or 0) + (kernel_ms["mesh_finish"] or 0))) if ms},
        "cpu_oracle_s_one_thread": oracle_s,
        "bit_identical_to_oracle": identical,
    }
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
