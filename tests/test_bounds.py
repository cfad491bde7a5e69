"""PredictBoundingBoxes on the device (SURVEY.md §8 f4, bepucuda_predict_bounding_boxes).

CPU: the oracle's restatement (oracle_predict_bounding_boxes) reproduces, bit for bit, the committed known-answer vectors generated from the reference's
own C# text (CapsuleWide / BoxWide / CylinderWide.GetBounds + BoundingBoxHelpers, transpiled: tests/golden/make_reference_bounds_vectors.py), the
same library's recorded answers on fresh random inputs (tests/golden/make_reference_fresh_vectors.py), and closed-form answers (a sphere at rest, sleep-candidacy counting).
GPU: the kernel is bit-identical to the oracle on random bodies of every supported shape, with the velocity callback, kinematic bodies, unsupported
shapes, and on the body state a solve leaves resident."""
import os

import numpy as np
import pytest

import bepuphysics2_b200 as bp
from bepuphysics2_b200 import native, scenes
from oracle import binding as ob

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DT = 1.0 / 60.0


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _identity_callback():
    integ = bp.IntegratorDesc.default()
    integ.gravity[0] = integ.gravity[1] = integ.gravity[2] = 0.0
    integ.linear_damping = 0.0
    integ.angular_damping = 0.0
    return integ


def _records(types, dims, margins, allow):
    n = types.shape[0]
    shapes = np.zeros(n, dtype=native.BODY_SHAPE_DTYPE)
    shapes["type"], shapes["a"], shapes["b"], shapes["c"] = types, dims[:, 0], dims[:, 1], dims[:, 2]
    shapes["minimum_speculative_margin"], shapes["maximum_speculative_margin"], shapes["allow_expansion_beyond_speculative_margin"] = margins[:, 0], margins[:, 1], allow
    activities = np.zeros(n, dtype=native.BODY_ACTIVITY_DTYPE)
    activities["sleep_threshold"] = 0.01
    activities["minimum_timesteps_under_threshold"] = 32
    return shapes, activities


def _bodies(q, pos, lin, ang):
    return scenes.make_bodies(pos, orientation=q, linear=lin, angular=ang, inverse_mass=np.ones(q.shape[0], dtype=np.float32),
                              inverse_inertia=np.tile(np.array([[1, 0, 1, 0, 0, 1]], dtype=np.float32), (q.shape[0], 1)))


def _oracle_on_inputs(types, dims, margins, allow, q, pos, lin, ang, dt):
    shapes, activities = _records(types, dims, margins, allow)
    # zero gravity and damping: the velocity callback is the identity ((v + 0) * 1), so the inputs are the "integrated" velocities the reference vectors use
    return ob.predict_bounding_boxes(_bodies(q, pos, lin, ang), shapes, activities, dt, _identity_callback())


def test_oracle_reproduces_the_reference_bounds_vectors_bit_for_bit(libs):
    golden = np.load(os.path.join(ROOT, "tests", "golden", "reference_bounds_vectors.npz"))
    for k in (0, 1):
        inputs = [golden["set%d_%s" % (k, name)] for name in ("types", "dims", "margins", "allow", "q", "pos", "lin", "ang")]
        got = _oracle_on_inputs(*inputs, float(golden["set%d_dt" % k]))
        assert (got[:, 7] == 1.0).all()
        assert np.array_equal(_bits(got[:, :7]), _bits(golden["set%d_out" % k])), "set %d" % k
        assert sorted(set(inputs[0].tolist())) == [0, 1, 2, 4]
    # the vectors reach the clamps: some margins sit on their bounds, some expansions are cut by the margin
    out, margins = golden["set0_out"], golden["set0_margins"]
    assert (out[:, 3] == margins[:, 0]).any() and (out[:, 3] == margins[:, 1]).any()


def test_oracle_matches_the_transpiled_reference_on_fresh_inputs(libs):
    """400 random bodies on another seed than the known-answer vectors; the transpiled library's bounds on them are recorded in
    tests/golden/reference_fresh_vectors.npz (tests/golden/make_reference_fresh_vectors.py)."""
    fresh = np.load(os.path.join(ROOT, "tests", "golden", "reference_fresh_vectors.npz"))
    inputs = [fresh["bounds_" + name] for name in ("types", "dims", "margins", "allow", "q", "pos", "lin", "ang")]
    assert inputs[0].shape == (400,)
    got = _oracle_on_inputs(*inputs, float(fresh["bounds_dt"]))
    assert np.array_equal(_bits(got[:, :7]), _bits(fresh["bounds_out"]))


def test_known_answers_and_sleep_candidacy(libs):
    integ = bp.IntegratorDesc.default()  # gravity (0, -10, 0), damping 0.03
    n = 4
    q = np.tile(np.array([[0, 0, 0, 1]], dtype=np.float32), (n, 1))
    pos = np.array([[1, 2, 3]] * n, dtype=np.float32)
    zero = np.zeros((n, 3), dtype=np.float32)
    types = np.array([0, 2, 7, -1], dtype=np.int32)
    dims = np.array([[0.5, 0, 0], [1, 2, 3], [1, 1, 1], [0, 0, 0]], dtype=np.float32)
    shapes, activities = _records(types, dims, np.tile(np.array([[0.0, 3.40282347e+38]], dtype=np.float32), (n, 1)), np.ones(n, dtype=np.int32))
    bodies = _bodies(q, pos, zero, zero)
    bodies[1, 16:23] = 0.0  # body 1 is kinematic: the callback leaves it alone, so it predicts no motion
    bounds = ob.predict_bounding_boxes(bodies, shapes, activities, DT, integ)
    # a sphere at rest: one frame of gravity (after damping) stretches the box downwards by |v| dt and the margin equals that displacement
    vy = np.float32(np.float32(-10.0 * np.float32(DT)) * np.float32(np.power(np.float32(0.97), np.float32(DT))))
    drop = np.float32(abs(vy) * np.float32(DT))
    assert np.allclose(bounds[0], [0.5, 1.5 - drop, 2.5, drop, 1.5, 2.5, 3.5, 1.0], rtol=0, atol=1e-6)
    # the axis-aligned kinematic box: exactly its half extents, zero margin
    assert np.array_equal(bounds[1], np.array([0, 0, 0, 0, 2, 4, 6, 1], dtype=np.float32))
    # a mesh (type 7) and a shapeless body: no bounds, activity still counted
    assert (bounds[2:] == 0).all()
    assert (activities["timesteps_under_threshold_count"] == 1).all() and (activities["sleep_candidate"] == 0).all()
    for _ in range(31):
        ob.predict_bounding_boxes(bodies, shapes, activities, DT, integ)
    assert (activities["timesteps_under_threshold_count"] == 32).all() and (activities["sleep_candidate"] == 1).all()
    activities["timesteps_under_threshold_count"] = 255  # saturates (PoseIntegrator.cs:L296)
    ob.predict_bounding_boxes(bodies, shapes, activities, DT, integ)
    assert (activities["timesteps_under_threshold_count"] == 255).all()
    bodies[:, 8] = 1.0  # moving again: |v|^2 = 1 > threshold
    ob.predict_bounding_boxes(bodies, shapes, activities, DT, integ)
    assert (activities["timesteps_under_threshold_count"] == 0).all() and (activities["sleep_candidate"] == 0).all()


def _random_world(rng, n):
    types = rng.choice([0, 1, 2, 4, 3, 5, -1], size=n, p=[0.2, 0.2, 0.25, 0.2, 0.05, 0.05, 0.05]).astype(np.int32)
    dims = rng.uniform(0.05, 3.0, size=(n, 3)).astype(np.float32)
    margins = np.stack([rng.choice([0.0, 0.01, 0.2], size=n), rng.choice([0.05, 1.0, 3.40282347e+38], size=n)], axis=1).astype(np.float32)
    shapes, activities = _records(types, dims, margins, rng.integers(0, 2, size=n).astype(np.int32))
    activities["sleep_threshold"] = rng.choice([-1.0, 0.01, 5.0], size=n)
    activities["minimum_timesteps_under_threshold"] = rng.integers(1, 40, size=n)
    activities["timesteps_under_threshold_count"] = rng.integers(0, 256, size=n)
    q = rng.normal(size=(n, 4))
    q = (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)
    bodies = _bodies(q, rng.uniform(-50, 50, size=(n, 3)).astype(np.float32), (rng.normal(size=(n, 3)) * rng.choice([0.0, 0.1, 5.0, 80.0], size=(n, 1))).astype(np.float32),
                     (rng.normal(size=(n, 3)) * rng.choice([0.0, 0.3, 10.0, 200.0], size=(n, 1))).astype(np.float32))
    bodies[rng.random(n) < 0.1, 16:23] = 0.0  # some kinematic bodies
    return bodies, shapes, activities


@pytest.mark.gpu
def test_device_bounds_are_bit_identical_to_the_oracle(libs):
    rng = np.random.default_rng(5)
    for integrate_kinematics in (0, 1):
        bodies, shapes, activities = _random_world(rng, 5000)
        integ = bp.IntegratorDesc.default()
        integ.integrate_velocity_for_kinematics = integrate_kinematics
        sim = bp.Simulation(integrator=integ)
        sim.add_bodies(bodies)
        ts = bp.CudaTimestepper(sim)
        try:
            ts.describe()
            ts.set_body_shapes(shapes)
            want_activities = activities.copy()
            for frame in range(3):  # the counters evolve over several frames
                want = ob.predict_bounding_boxes(bodies, shapes, want_activities, DT, integ)
                got = ts.predict_bounding_boxes(DT, activities)
                assert np.array_equal(_bits(got), _bits(want)), "frame %d" % frame
                assert np.array_equal(activities.view(np.uint8), want_activities.view(np.uint8))
            assert (got[:, 7] == np.isin(shapes["type"], [0, 1, 2, 4])).all()
            with pytest.raises(bp.BepuCudaError):
                ts.set_body_shapes(shapes[:10])
                ts.predict_bounding_boxes(DT, activities)
        finally:
            ts.close()


@pytest.mark.gpu
def test_device_bounds_on_the_state_a_solve_leaves_resident(libs):
    """DefaultTimestepper order: ... Solve | next frame: PredictBoundingBoxes. The bounds come from the bodies the solve left on the device."""
    from tests import util

    scene = scenes.shape_pile(3000, seed=4)
    a = util.make_sim(scene, substeps=2, velocity_iterations=2)
    b = util.make_sim(scene, substeps=2, velocity_iterations=2)
    rng = np.random.default_rng(9)
    _, shapes, activities = _random_world(rng, a.body_count)
    ob.solve(a, DT)
    want_activities = activities.copy()
    want = ob.predict_bounding_boxes(a.bodies, shapes, want_activities, DT, a.integrator)
    ts = bp.CudaTimestepper(b, strict_fp=True)
    try:
        ts.describe()
        ts.set_body_shapes(shapes)
        ts.solve_device_only(DT)
        got = ts.predict_bounding_boxes(DT, activities)
    finally:
        ts.close()
    assert np.array_equal(_bits(got), _bits(want))
    assert np.array_equal(activities.view(np.uint8), want_activities.view(np.uint8))
