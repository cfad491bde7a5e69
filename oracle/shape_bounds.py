"""ORACLE — test infrastructure only. ctypes loader for oracle/libbepu_oracle_shapes.so (bepu_oracle_shapes.cpp): PredictBoundingBoxes for every
built-in shape type, restated sequentially in the reference's loop order. Compiled with the flags of oracle/Makefile (-ffp-contract=off)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libbepu_oracle_shapes.so")
SOURCES = [os.path.join(HERE, f) for f in ("bepu_oracle_shapes.cpp", "bepu_math.h")]
_LIB = None


def build(force=False):
    if force or not os.path.exists(LIB) or any(os.path.getmtime(s) > os.path.getmtime(LIB) for s in SOURCES):
        cmd = ["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-march=x86-64-v3", "-Wall", "-Wno-unused-function", "-Wno-psabi",
               "-shared", "-o", LIB, SOURCES[0]]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("shape-bounds oracle build failed:\n" + r.stdout)
    return LIB


def load():
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(build())
        _LIB.oracle_predict_bounding_boxes_collidables.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_float, C.c_float,
                                                                   C.c_int32, C.c_void_p]
    return _LIB


def predict_bounding_boxes_collidables(bodies, collidables, activities, library, dt, integrator):
    """bodies[n, 32] (BodyDynamics records), collidables (BODY_COLLIDABLE_DTYPE), activities (BODY_ACTIVITY_DTYPE, updated in place), library
    (bepuphysics2_b200.ShapeLibrary). Returns bounds[n, 8] = {min.xyz, speculative margin, max.xyz, valid}."""
    lib = load()
    bodies = np.ascontiguousarray(bodies, dtype=np.float32).reshape(-1, 32)
    n = bodies.shape[0]
    assert collidables.shape[0] == n and activities.shape[0] == n and collidables.dtype.itemsize == 16 and activities.dtype.itemsize == 8
    assert activities.flags["C_CONTIGUOUS"]
    collidables = np.ascontiguousarray(collidables)
    desc = library.desc()
    bounds = np.zeros((max(n, 1), 8), dtype=np.float32)
    gravity = (C.c_float * 3)(*integrator.gravity)
    rc = lib.oracle_predict_bounding_boxes_collidables(n, bodies.ctypes.data, collidables.ctypes.data, activities.ctypes.data, C.addressof(desc), dt, gravity,
                                                       integrator.linear_damping, integrator.angular_damping, int(integrator.integrate_velocity_for_kinematics), bounds.ctypes.data)
    if rc != 0:
        raise ValueError("oracle_predict_bounding_boxes_collidables: a shape index is out of range")
    return bounds[:n]
