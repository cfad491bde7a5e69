"""Pins the hand-written oracle (oracle/*.h) to the REFERENCE'S OWN C# TEXT.

The reference cannot be built here (no .NET). Its constraint functions, wide math and pose integration are straight-line code, so
oracle/ref_transpile/cs2cpp.py transpiles those sources mechanically (syntax only; every operator and call is the C# text's, in its order) into
oracle/_ref/libbepu_ref.so, compiled without FMA contraction like RyuJIT's Vector<float> code. Two layers of checks, all BIT FOR BIT:

  * committed known-answer vectors (tests/golden/reference_vectors.npz, generated from the transpiled reference by
    tests/golden/make_reference_vectors.py): every one of the 44 constraint types x {WarmStart, Solve, IncrementallyUpdateForSubstep}, the four
    PoseIntegration functions, and 38 chains of 1000 x (WarmStart; Solve) on the reference's constraint micro-benchmark inputs
    (DemoBenchmarks/*ConstraintBenchmarks*.cs);
  * fresh inputs (tests/golden/reference_fresh_vectors.npz, recorded from the same library by tests/golden/make_reference_fresh_vectors.py):
    32 more samples per type on other seeds, degenerate lanes among them.
Both files are committed, so the checks run without the reference tree.

What stays outside the pin: the solver driver (substep loop, batch order, integration responsibilities, gather/scatter, the TypeProcessor bundle
loops), which is generic / unsafe C# the transpiler does not cover; tests/test_oracle.py holds those to closed-form answers.
TEST INFRASTRUCTURE: nothing in the product loads either library."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import binding as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FP = C.POINTER(C.c_float)
DT = 1.0 / 240.0


def _ptr(a):
    return a.ctypes.data_as(FP)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


@pytest.fixture(scope="module")
def oracle(libs):
    lib = ob.load()
    lib.oracle_eval_lane.argtypes = [C.c_int32, C.c_int32, FP, C.c_float, FP, FP, FP, C.c_int32]
    lib.oracle_eval_integration.argtypes = [C.c_int32, FP, FP]
    return lib


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))


def test_golden_vectors_cover_every_registered_type(oracle, golden):
    registered = sorted(t for t in range(64) if ob.type_info(t) is not None)
    in_file = sorted(int(k[5:7]) for k in golden.files if k.startswith("lane_") and k.endswith("_states"))
    assert registered == in_file and len(registered) == 44


def test_oracle_reproduces_the_reference_constraint_functions_bit_for_bit(oracle, golden):
    checked = 0
    for type_id in sorted(t for t in range(64) if ob.type_info(t) is not None):
        key = "lane_%02d_" % type_id
        states, vel, imp, pre = (golden[key + n] for n in ("states", "velocities", "impulses", "prestep"))
        bodies, prestep_rows, impulse_rows = ob.type_info(type_id)
        assert states.shape[1:] == (bodies, 14) and imp.shape[1] == impulse_rows and pre.shape[1] == prestep_rows
        for i in range(states.shape[0]):
            for stage in (0, 1, 2):
                v, a, p = vel[i].copy(), imp[i].copy(), pre[i].copy()
                st = np.ascontiguousarray(states[i])
                assert oracle.oracle_eval_lane(type_id, stage, _ptr(st), DT, _ptr(p), _ptr(a), _ptr(v), 1) == 0
                what = "type %d stage %d sample %d" % (type_id, stage, i)
                assert np.array_equal(_bits(v), _bits(golden[key + "out%d_velocities" % stage][i])), what + ": velocities"
                assert np.array_equal(_bits(a), _bits(golden[key + "out%d_impulses" % stage][i])), what + ": accumulated impulses"
                assert np.array_equal(_bits(p), _bits(golden[key + "out%d_prestep" % stage][i])), what + ": prestep"
                checked += 1
        # the vectors exercise the functions: WarmStart and Solve moved the velocities
        assert not np.array_equal(golden[key + "out1_velocities"], vel)
    assert checked == 44 * 3 * 6


def test_oracle_reproduces_the_reference_pose_integration_bit_for_bit(oracle, golden):
    """PoseIntegration.Integrate (custom Sin/Cos, normalisation, |w| <= 1e-15 fallback), RotateInverseInertia, IntegrateAngularVelocityConserveMomentum,
    ...WithGyroscopicTorque (BepuPhysics/PoseIntegrator.cs:L146-253)."""
    for op in range(4):
        ins, outs = golden["integration_%d_in" % op], golden["integration_%d_out" % op]
        for i in range(ins.shape[0]):
            got = np.zeros(outs.shape[1], dtype=np.float32)
            assert oracle.oracle_eval_integration(op, _ptr(np.ascontiguousarray(ins[i])), _ptr(got)) == 0
            assert np.array_equal(_bits(got), _bits(outs[i])), "integration function %d sample %d" % (op, i)


def test_oracle_reproduces_the_reference_benchmark_chains_bit_for_bit(oracle, golden):
    """DemoBenchmarks/{One,Two,Three,Four}BodyConstraintBenchmarks[Deep].cs: 1000 x (WarmStart; Solve) at dt = 1/60 from rest on the benchmark's own
    prestep data; a chain amplifies any difference in a single evaluation, and exercises warm starting with the solver's own accumulated impulses."""
    names = list(golden["bench_names"])
    assert len(names) >= 30
    for n, name in enumerate(names):
        k = "bench_%02d_" % n
        tid = int(golden[k + "type"])
        st, p = np.ascontiguousarray(golden[k + "states"]), golden[k + "prestep"].copy()
        v, a = np.zeros_like(golden[k + "out_velocities"]), np.zeros_like(golden[k + "out_impulses"])
        for _ in range(1000):
            oracle.oracle_eval_lane(tid, 0, _ptr(st), 1.0 / 60.0, _ptr(p), _ptr(a), _ptr(v), 1)
            oracle.oracle_eval_lane(tid, 1, _ptr(st), 1.0 / 60.0, _ptr(p), _ptr(a), _ptr(v), 1)
        assert np.isfinite(v).all(), name
        assert np.array_equal(_bits(v), _bits(golden[k + "out_velocities"])), name + ": velocities after 1000 iterations"
        assert np.array_equal(_bits(a), _bits(golden[k + "out_impulses"])), name + ": accumulated impulses after 1000 iterations"


@pytest.fixture(scope="module")
def fresh():
    """The transpiled reference's answers on the fresh inputs, recorded by tests/golden/make_reference_fresh_vectors.py."""
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_fresh_vectors.npz"))


def test_transpiled_reference_covers_all_types_and_reproduces_the_committed_vectors(oracle, golden, fresh):
    assert sorted(fresh["covered_types"].tolist()) == sorted(t for t in range(64) if ob.type_info(t) is not None)
    # both committed files come from the same library (regenerate them together with tests/golden/make_reference_vectors.py and
    # tests/golden/make_reference_fresh_vectors.py)
    assert np.array_equal(_bits(fresh["committed_lane_07_out1_velocities"]), _bits(golden["lane_07_out1_velocities"][0]))


def test_oracle_matches_the_transpiled_reference_on_fresh_inputs(oracle, fresh):
    """Every type, every stage, 16 fresh samples per type (other seeds than the committed vectors), plus degenerate lanes: zero velocities and
    impulses, identical poses, a kinematic partner (zero inverse mass and inertia). An output the file leaves out is the reference's input, unchanged."""
    types = fresh["lane_types"].tolist()
    assert types == sorted(t for t in range(64) if ob.type_info(t) is not None)
    floats = {t: dict(zip(("states", "velocities", "impulses", "prestep"), (b * 14, b * 6, d, p))) for t, (b, p, d) in ((t, ob.type_info(t)) for t in types)}

    def split(name, among):
        """The [16, floats per sample] blocks of the types `among` from the flat array lane_<name>."""
        flat, out, at = fresh["lane_" + name], {}, 0
        for t in among:
            n = 16 * floats[t][name.split("_")[-1]]
            out[t] = flat[at:at + n].reshape(16, -1)
            at += n
        assert at == flat.size, name
        return out

    given = {n: split(n, types) for n in ("states", "velocities", "impulses", "prestep")}
    want = {}
    for stage in (0, 1, 2):
        for n in ("velocities", "impulses", "prestep"):
            key = "lane_out%d_%s_types" % (stage, n)
            changed = split("out%d_%s" % (stage, n), fresh[key].tolist()) if key in fresh.files else {}
            want[(stage, n)] = {t: changed.get(t, given[n][t]) for t in types}
    for type_id in types:
        for i in range(16):
            st = np.ascontiguousarray(given["states"][type_id][i])
            for stage in (0, 1, 2):
                got = {n: given[n][type_id][i].copy() for n in ("velocities", "impulses", "prestep")}
                assert oracle.oracle_eval_lane(type_id, stage, _ptr(st), DT, _ptr(got["prestep"]), _ptr(got["impulses"]), _ptr(got["velocities"]), 1) == 0
                for n in got:
                    assert np.array_equal(_bits(got[n]), _bits(want[(stage, n)][type_id][i])), "type %d stage %d sample %d: %s" % (type_id, stage, i, n)
