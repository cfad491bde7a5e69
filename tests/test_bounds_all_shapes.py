"""PredictBoundingBoxes for every built-in shape type (bepucuda_set_shape_library / bepucuda_set_body_collidables).

CPU: the oracle's sequential restatement (oracle/bepu_oracle_shapes.cpp) and the CUDA arithmetic compiled for the host
(tests/device_on_host/shape_bounds_on_host.cpp, replaying the kernels' reduction order) reproduce, bit for bit, the committed vectors generated from
the reference's own C# text (tests/golden/make_reference_shape_bounds_vectors.py), including the signed-zero fixture; closed-form answers hold.
GPU: the kernels are bit-identical to the oracle on random worlds of every type, over several frames, at every hull width, with large compounds, a
mesh spread over several CTAs, the signed-zero fixture and the state a solve leaves resident; the set calls reject malformed input."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import bepuphysics2_b200 as bp
from bepuphysics2_b200 import native, scenes
from bepuphysics2_b200.native import ShapeLibrary, typed_index
from oracle import binding as ob
from oracle import shape_bounds as osb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.join(ROOT, "tests", "device_on_host")
CSRC = os.path.join(ROOT, "bepuphysics2_b200", "csrc")
DT = 1.0 / 60.0
FP = C.POINTER(C.c_float)
LIBRARY_FIELDS = ("spheres", "capsules", "boxes", "triangles", "cylinders", "hull_points", "hulls", "compound_children", "compounds", "big_compounds", "mesh_triangles", "meshes")
GOLDEN_SETS = ("w4", "w8", "w16", "zero")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _no_callback():
    """Integrator settings under which the oracle leaves the velocity alone: every test body is kinematic and kinematics are not integrated, so the
    inputs are the post-callback velocities the vectors were generated with (an identity callback would turn -0 into +0)."""
    integ = bp.IntegratorDesc.default()
    integ.integrate_velocity_for_kinematics = 0
    return integ


def _inputs(golden, s):
    library = ShapeLibrary(hull_bundle_width=int(golden[s + "_width"]), **{f: golden[s + "_lib_" + f] for f in LIBRARY_FIELDS})
    return [library] + [np.ascontiguousarray(golden["%s_%s" % (s, k)]) for k in ("shape", "margins", "allow", "q", "pos", "lin", "ang")] + [float(golden[s + "_dt"])]


def _collidables(shape, margins, allow):
    c = np.zeros(shape.shape[0], dtype=native.BODY_COLLIDABLE_DTYPE)
    c["shape"], c["minimum_speculative_margin"], c["maximum_speculative_margin"], c["allow_expansion_beyond_speculative_margin"] = shape, margins[:, 0], margins[:, 1], allow
    return c


def _oracle(library, shape, margins, allow, q, pos, lin, ang, dt):
    n = shape.shape[0]
    bodies = scenes.make_bodies(pos, orientation=q, linear=lin, angular=ang)  # kinematic: zero inverse mass and inertia
    activities = np.zeros(n, dtype=native.BODY_ACTIVITY_DTYPE)
    return osb.predict_bounding_boxes_collidables(bodies, _collidables(shape, margins, allow), activities, library, dt, _no_callback())


@pytest.fixture(scope="module")
def on_host():
    lib = os.path.join(HERE, "libshape_bounds_on_host.so")
    srcs = [os.path.join(HERE, "shape_bounds_on_host.cpp"), os.path.join(HERE, "stubs", "cuda_runtime.h")] + [os.path.join(CSRC, f) for f in ("bepu_device_math.cuh", "bepu_bounds_math.cuh", "bepu_shape_bounds_math.cuh")]
    if not os.path.exists(lib) or any(os.path.getmtime(s) > os.path.getmtime(lib) for s in srcs):
        subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-march=x86-64-v3", "-Wall", "-Wno-unused-function", "-I", os.path.join(HERE, "stubs"),
                               "-I", CSRC, "-shared", "-fPIC", "-o", lib, srcs[0]])
    dev = C.CDLL(lib)
    dev.shape_bounds_on_host.argtypes = [C.c_void_p, C.c_uint32, FP, C.c_int32, FP, FP, FP, FP, C.c_float, C.c_int32, FP]
    return dev


def _on_host(dev, library, shape, margins, allow, q, pos, lin, ang, dt, mesh_chunk=64):
    desc = library.desc()
    out = np.zeros((shape.shape[0], 7), dtype=np.float32)
    p = lambda a: a.ctypes.data_as(FP)
    for i in range(shape.shape[0]):
        if dev.shape_bounds_on_host(C.addressof(desc), int(shape[i]), p(margins[i]), int(allow[i]), p(q[i]), p(pos[i]), p(lin[i]), p(ang[i]), dt, mesh_chunk, p(out[i])) != 0:
            out[i] = 0.0
    return out


def test_oracle_reproduces_the_reference_shape_bounds_vectors_bit_for_bit(libs):
    golden = np.load(os.path.join(ROOT, "tests", "golden", "reference_shape_bounds_vectors.npz"))
    for s in GOLDEN_SETS:
        inputs = _inputs(golden, s)
        got = _oracle(*inputs)
        assert np.array_equal(_bits(got[:, :7]), _bits(golden[s + "_out"])), s
        types = (inputs[1] >> 24) & 0x7F
        exists = (inputs[1] >> 31) == 1
        assert ((got[:, 7] == 1) == (exists & (types <= 8))).all(), s
        if s != "zero":
            assert set(types[exists & (types <= 8)].tolist()) == set(range(9)), s
            children = inputs[0].compound_children["shape"]
            assert set(((children >> 24) & 0x7F).tolist()) == set(range(6)), "compounds mix all six convex child types"
    # the vectors reach the clamps: margins on both bounds, fast spins past pi/3
    out = np.concatenate([golden[s + "_out"] for s in ("w4", "w8", "w16")])
    margins = np.concatenate([golden[s + "_margins"] for s in ("w4", "w8", "w16")])
    assert (out[:, 3] == margins[:, 0]).any() and (out[:, 3] == margins[:, 1]).any()
    assert (np.linalg.norm(golden["w8_ang"], axis=1) * float(golden["w8_dt"]) > np.pi / 3).any()
    # the signed-zero fixture: the sign of the zero each fold keeps reaches max.z, and both signs occur
    zmax = golden["zero_out"][:, 6]
    assert (zmax == 0).all() and np.signbit(zmax).any() and not np.signbit(zmax).all()


def test_device_source_reproduces_the_reference_shape_bounds_vectors_bit_for_bit(on_host):
    """csrc/bepu_shape_bounds_math.cuh compiled for the host, with the kernels' combining order replayed (mesh chunks of 64 and of 8192 triangles)."""
    golden = np.load(os.path.join(ROOT, "tests", "golden", "reference_shape_bounds_vectors.npz"))
    for s in GOLDEN_SETS:
        for chunk in (64, 8192):
            got = _on_host(on_host, *_inputs(golden, s), mesh_chunk=chunk)
            assert np.array_equal(_bits(got), _bits(golden[s + "_out"])), "%s, chunk %d" % (s, chunk)


def _single(library, shape, q=(0, 0, 0, 1), pos=(0, 0, 0), lin=(0, 0, 0), ang=(0, 0, 0), margins=(0.0, 3.40282347e+38), allow=1, dt=DT):
    a = lambda v, k: np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(1, k))
    return (library, np.array([shape], dtype=np.uint32), a(margins, 2), np.array([allow], dtype=np.int32), a(q, 4), a(pos, 3), a(lin, 3), a(ang, 3), dt)


def test_closed_form_answers(libs, on_host):
    rng = np.random.default_rng(3)
    evaluators = (lambda *x: _oracle(*x)[:, :7], lambda *x: _on_host(on_host, *x))
    points = rng.uniform(-2, 2, (37, 3)).astype(np.float32)
    pos = np.float32([1.5, -2.25, 3.0])
    per_width = []
    q = rng.normal(size=4).astype(np.float32)
    q /= np.linalg.norm(q)
    for w in (4, 8, 16):
        lib = ShapeLibrary(hull_points=scenes.bundle_hull_points(points, w), hull_bundle_width=w, hulls=[(0, (37 + w - 1) // w)])
        for ev in evaluators:
            got = ev(*_single(lib, typed_index(5, 0), pos=pos))[0]
            # at identity orientation and rest the box is exactly position + the min / max of the points (x * 1 + y * 0 + z * 0 is exact)
            assert np.array_equal(got[[0, 1, 2]], pos + points.min(axis=0)) and np.array_equal(got[[4, 5, 6]], pos + points.max(axis=0))
            assert got[3] == 0.0
            per_width.append(ev(*_single(lib, typed_index(5, 0), q=q, lin=(1, 2, 3), ang=(4, 5, 6)))[0])
    # hull bounds are value-equal across widths (only the sign of a tied zero may depend on W)
    assert all(np.array_equal(per_width[0], x) for x in per_width[1:])
    # one child at the local identity pose == that child's own bounds; a big compound == the compound with the same children
    base = scenes.shape_library(rng, hull_width=8, primitives=4, hulls=2, compounds=0, big_compounds=0)
    children = np.zeros(6, dtype=native.COMPOUND_CHILD_DTYPE)
    children["local_orientation"][:, 3] = 1.0
    children["shape"] = typed_index(np.arange(6), np.zeros(6))
    lib = ShapeLibrary(**{f: getattr(base, f) for f in LIBRARY_FIELDS if f not in ("compound_children", "compounds", "big_compounds")}, hull_bundle_width=8,
                       compound_children=children, compounds=[(k, 1) for k in range(6)] + [(0, 6)], big_compounds=[(0, 6)])
    q = rng.normal(size=4).astype(np.float32)
    motion = dict(q=q / np.linalg.norm(q), pos=(3, -1, 2), lin=(0.5, -2, 1), ang=(0.3, 9, -2), margins=(0.01, 1.0), allow=0)
    for ev in evaluators:
        for t in range(6):
            assert np.array_equal(ev(*_single(lib, typed_index(6, t), **motion)), ev(*_single(lib, typed_index(t, 0), **motion))), "child type %d" % t
        assert np.array_equal(ev(*_single(lib, typed_index(7, 0), **motion)), ev(*_single(lib, typed_index(6, 6), **motion)))
    # a mesh at identity, at rest, zero minimum margin: exactly position + the min / max of scale * vertices
    tri = rng.uniform(-3, 3, (300, 9)).astype(np.float32)
    s = np.float32([0.5, 2.0, 1.25])
    lib = ShapeLibrary(mesh_triangles=tri, meshes=[(0, 300, tuple(s))])
    scaled = (tri.reshape(-1, 3) * s).astype(np.float32)
    for ev in evaluators:
        got = ev(*_single(lib, typed_index(8, 0), pos=pos))[0]
        assert np.array_equal(got[[0, 1, 2]], pos + scaled.min(axis=0)) and np.array_equal(got[[4, 5, 6]], pos + scaled.max(axis=0)) and got[3] == 0.0


# ---------------------------------------------------------------------------------------------------------------------------------------------------
def _device_vs_oracle(world, integ, frames=3, bodies=None):
    """Runs `frames` predictions on the device and the oracle from the same activities; returns the last device bounds."""
    bodies = world["bodies"] if bodies is None else bodies
    sim = bp.Simulation(integrator=integ)
    sim.add_bodies(bodies)
    ts = bp.CudaTimestepper(sim)
    try:
        ts.describe()
        ts.set_shape_library(world["library"])
        ts.set_body_collidables(world["collidables"])
        got_act, want_act = world["activities"].copy(), world["activities"].copy()
        for frame in range(frames):
            want = osb.predict_bounding_boxes_collidables(bodies, world["collidables"], want_act, world["library"], DT, integ)
            got = ts.predict_bounding_boxes(DT, got_act)
            assert np.array_equal(_bits(got), _bits(want)), "frame %d: %d rows differ" % (frame, int((_bits(got) != _bits(want)).any(axis=1).sum()))
            assert np.array_equal(got_act.view(np.uint8), want_act.view(np.uint8))
        return got
    finally:
        ts.close()


@pytest.mark.gpu
def test_device_matches_the_oracle_on_mixed_worlds(libs):
    for integrate_kinematics in (0, 1):
        for w in (4, 8, 16):
            world = scenes.shape_world(4000, seed=10 + w + integrate_kinematics, hull_width=w, mesh_triangle_counts=(300, 900))
            integ = bp.IntegratorDesc.default()
            integ.integrate_velocity_for_kinematics = integrate_kinematics
            got = _device_vs_oracle(world, integ)
            shape = world["collidables"]["shape"]
            assert (got[:, 7] == (((shape >> 31) == 1) & (((shape >> 24) & 0x7F) <= 8))).all()


@pytest.mark.gpu
def test_device_large_compounds_and_multi_cta_meshes(libs):
    rng = np.random.default_rng(17)
    library = scenes.shape_library(rng, hull_width=8, compounds=6, big_compounds=3, compound_children=(900, 1100), mesh_triangle_counts=(3 * 8192 + 17, 100_000, 8192))
    world = scenes.shape_world(600, seed=18, library=library, type_weights={5: 1, 6: 2, 7: 2, 8: 2, 0: 1})
    _device_vs_oracle(world, bp.IntegratorDesc.default(), frames=2)


@pytest.mark.gpu
def test_device_signed_zero_fixture(libs):
    golden = np.load(os.path.join(ROOT, "tests", "golden", "reference_shape_bounds_vectors.npz"))
    library, shape, margins, allow, q, pos, lin, ang, dt = _inputs(golden, "zero")
    bodies = scenes.make_bodies(pos, orientation=q, linear=lin, angular=ang)
    sim = bp.Simulation(integrator=_no_callback())
    sim.add_bodies(bodies)
    ts = bp.CudaTimestepper(sim)
    try:
        ts.describe()
        ts.set_shape_library(library)
        ts.set_body_collidables(_collidables(shape, margins, allow))
        got = ts.predict_bounding_boxes(dt, np.zeros(shape.shape[0], dtype=native.BODY_ACTIVITY_DTYPE))
    finally:
        ts.close()
    assert np.array_equal(_bits(got[:, :7]), _bits(golden["zero_out"]))


@pytest.mark.gpu
def test_device_on_the_state_a_solve_leaves_resident(libs):
    from tests import util

    scene = scenes.shape_pile(3000, seed=4)
    a = util.make_sim(scene, substeps=2, velocity_iterations=2)
    b = util.make_sim(scene, substeps=2, velocity_iterations=2)
    world = scenes.shape_world(a.body_count, seed=9, mesh_triangle_counts=(500,))
    ob.solve(a, DT)
    want_act = world["activities"].copy()
    want = osb.predict_bounding_boxes_collidables(a.bodies, world["collidables"], want_act, world["library"], DT, a.integrator)
    ts = bp.CudaTimestepper(b, strict_fp=True)
    try:
        ts.describe()
        ts.set_shape_library(world["library"])
        ts.set_body_collidables(world["collidables"])
        ts.solve_device_only(DT)
        got_act = world["activities"].copy()
        got = ts.predict_bounding_boxes(DT, got_act)
    finally:
        ts.close()
    assert np.array_equal(_bits(got), _bits(want))
    assert np.array_equal(got_act.view(np.uint8), want_act.view(np.uint8))


@pytest.mark.gpu
def test_set_calls_reject_malformed_input_and_legacy_mode_returns(libs):
    world = scenes.shape_world(200, seed=2, mesh_triangle_counts=(50,))
    good = world["library"]
    sim = bp.Simulation()
    sim.add_bodies(world["bodies"])
    ts = bp.CudaTimestepper(sim)

    def lib_with(**change):
        kw = {f: getattr(good, f) for f in LIBRARY_FIELDS}
        kw["hull_bundle_width"] = good.hull_bundle_width
        kw.update(change)
        return ShapeLibrary(**kw)

    try:
        ts.describe()
        with pytest.raises(bp.BepuCudaError):  # collidables before any library
            ts.set_body_collidables(world["collidables"])
        bad_children = good.compound_children.copy()
        bad_children["shape"][0] = typed_index(6, 0)  # a compound child that is not convex
        out_of_range = good.compound_children.copy()
        out_of_range["shape"][0] = typed_index(0, len(good.spheres))
        hulls, compounds, meshes = good.hulls.copy(), good.compounds.copy(), good.meshes.copy()
        hulls["bundle_count"][0] = 0
        compounds["child_count"][0] = 0
        meshes["triangle_count"][0] = 0
        beyond = good.meshes.copy()
        beyond["triangle_count"][0] = len(good.mesh_triangles) + 1
        for what in (dict(hull_bundle_width=6), dict(hulls=hulls), dict(compounds=compounds), dict(meshes=meshes), dict(meshes=beyond), dict(compound_children=bad_children),
                     dict(compound_children=out_of_range)):
            with pytest.raises(bp.BepuCudaError):
                ts.set_shape_library(lib_with(**what))
        ts.set_shape_library(good)
        bad = world["collidables"].copy()
        bad["shape"][0] = typed_index(5, len(good.hulls))
        with pytest.raises(bp.BepuCudaError):
            ts.set_body_collidables(bad)
        ts.set_body_collidables(world["collidables"])
        assert ts.predict_bounding_boxes(DT, world["activities"].copy())[:, 7].any()
        # set_body_shapes switches back to the primitive-only path: types 3 / 5 / 7 get valid = 0 again
        shapes = np.zeros(200, dtype=native.BODY_SHAPE_DTYPE)
        shapes["type"] = np.resize([0, 3, 5, 7], 200)
        shapes["a"] = 1.0
        ts.set_body_shapes(shapes)
        got = ts.predict_bounding_boxes(DT, world["activities"].copy())
        assert (got[:, 7] == (shapes["type"] == 0)).all()
    finally:
        ts.close()
