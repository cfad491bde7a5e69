"""Generates tests/golden/reference_fresh_vectors.npz: the transpiled reference's answers on the "fresh" inputs of
tests/test_oracle_pinned_to_reference.py and tests/test_bounds.py (other seeds than reference_vectors.npz / reference_bounds_vectors.npz, plus
degenerate lanes), so that the oracle is held to the reference on them without the reference tree. Needs the reference sources (or a prebuilt
oracle/_ref/libbepu_ref.so); set BEPU_REFERENCE_ROOT to the reference's checkout.

    python tests/golden/make_reference_fresh_vectors.py

Stored: the types the transpiled library covers; per constraint type (lane_types), SAMPLES samples of inputs (lane_states, lane_velocities,
lane_impulses, lane_prestep) and the outputs of stage s = WarmStart / Solve / IncrementallyUpdateForSubstep (lane_out<s>_<input name>), each as ONE
flat float32 array: the types' [SAMPLES, floats per sample] blocks back to back in lane_types order. An output that is bit for bit its input
(WarmStart leaves the prestep alone, for instance) is stored only for the types where it is not (lane_out<s>_<name>_types); the others are checked
against the input. Then the library's Solve output on the first lane_07 sample of reference_vectors.npz, and 400 random convex bodies with their bounds.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_transpile"))
import build_ref  # noqa: E402
import make_reference_bounds_vectors as bounds_gen  # noqa: E402

FP = C.POINTER(C.c_float)
DT = 1.0 / 240.0
BOUNDS_DT = 1.0 / 60.0
SAMPLES = 16
PATH = os.path.join(ROOT, "tests", "golden", "reference_fresh_vectors.npz")


def ptr(a):
    return a.ctypes.data_as(FP)


def fresh_lane_inputs():
    """type id -> (states[n, bodies, 14], velocities[n, bodies, 6], impulses[n, impulse rows], prestep[n, prestep rows]): SAMPLES samples per type,
    every eighth from 5 on with zero velocities and impulses, from 6 on a kinematic partner (zero inverse mass and inertia), from 7 on identical poses."""
    from oracle import binding as ob
    from tests.test_device_source_on_host import _prestep_samples, _random_states

    samples = _prestep_samples()
    rng = np.random.default_rng(991)
    out = {}
    for type_id in sorted(samples):
        bodies, _, impulse_rows = ob.type_info(type_id)
        rows = []
        for n, prestep in enumerate(samples[type_id][:SAMPLES]):
            states = _random_states(rng, bodies)
            vel = rng.normal(0, 1.5, (bodies, 6)).astype(np.float32)
            imp = np.abs(rng.normal(0, 0.2, impulse_rows)).astype(np.float32)
            if n % 8 == 5:
                vel[:] = 0
                imp[:] = 0
            if n % 8 == 6 and bodies > 1:
                states[1, 7:14] = 0
            if n % 8 == 7:
                states[:, 3:7] = (0, 0, 0, 1)
            rows.append((states, vel, imp, prestep))
        out[type_id] = tuple(np.stack(parts) for parts in zip(*rows))
    return out


def main():
    lib = C.CDLL(build_ref.build())
    lib.ref_eval_lane.argtypes = [C.c_int32, C.c_int32, FP, C.c_float, FP, FP, FP, C.c_int32]
    lib.ref_covered_types.argtypes = [C.POINTER(C.c_int32), C.c_int32]
    out = {}
    ids = (C.c_int32 * 64)()
    out["covered_types"] = np.array(sorted(ids[:lib.ref_covered_types(ids, 64)]), dtype=np.int32)
    lanes = fresh_lane_inputs()
    blocks = {}  # array name -> [(type id, block)]
    for type_id, (states, vel, imp, pre) in lanes.items():
        for name, given in (("states", states), ("velocities", vel), ("impulses", imp), ("prestep", pre)):
            blocks.setdefault(name, []).append((type_id, given))
        for stage in (0, 1, 2):
            v, a, p = vel.copy(), imp.copy(), pre.copy()
            for i in range(states.shape[0]):
                assert lib.ref_eval_lane(type_id, stage, ptr(np.ascontiguousarray(states[i])), DT, ptr(p[i]), ptr(a[i]), ptr(v[i]), 1) == 0
            for name, result, given in (("velocities", v, vel), ("impulses", a, imp), ("prestep", p, pre)):
                if not np.array_equal(result.view(np.uint32), given.view(np.uint32)):
                    blocks.setdefault("out%d_%s" % (stage, name), []).append((type_id, result))
    out["lane_types"] = np.array(sorted(lanes), dtype=np.int32)
    for name, typed in blocks.items():
        out["lane_" + name] = np.concatenate([b.ravel() for _, b in typed])
        if name.startswith("out"):
            out["lane_%s_types" % name] = np.array([t for t, _ in typed], dtype=np.int32)
    committed = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))
    v, a, p = (committed["lane_07_" + n][0].copy() for n in ("velocities", "impulses", "prestep"))
    assert lib.ref_eval_lane(7, 1, ptr(np.ascontiguousarray(committed["lane_07_states"][0])), DT, ptr(p), ptr(a), ptr(v), 1) == 0
    out["committed_lane_07_out1_velocities"] = v
    inputs = bounds_gen.make_inputs(np.random.default_rng(77), 400)
    for name, a in zip(("types", "dims", "margins", "allow", "q", "pos", "lin", "ang"), inputs):
        out["bounds_" + name] = a
    out["bounds_dt"] = np.float32(BOUNDS_DT)
    out["bounds_out"] = bounds_gen.evaluate(bounds_gen.load_ref(), *inputs, BOUNDS_DT)
    np.savez_compressed(PATH, **out)
    print("wrote %s (%d bytes): %d constraint types x 3 stages, %d bounds samples" % (PATH, os.path.getsize(PATH), len(out["covered_types"]), inputs[0].shape[0]))


if __name__ == "__main__":
    main()
