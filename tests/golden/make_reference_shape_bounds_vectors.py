"""Generates tests/golden/reference_shape_bounds_vectors.npz: known-answer vectors for PredictBoundingBoxes over every built-in shape type, produced
by the REFERENCE'S OWN C# text where the transpiler carries it (TriangleWide / CapsuleWide / BoxWide / CylinderWide.GetBounds, BoundingBoxHelpers,
Matrix3x3Wide, Vector3Wide, QuaternionEx.ConcatenateWithoutOverlap / TransformWithoutOverlap, Matrix3x3.CreateFromQuaternion / Transform; see
oracle/ref_transpile/shape_bounds_ref.py) and by glue over those calls that cites the C# it follows where it does not (the hull's point-bundle walk,
the compound child loop, the mesh triangle loop: ref_shape_bounds in oracle/ref_transpile/shape_bounds_harness.cpp). Run where /root/reference exists; the file is committed
so that the check runs anywhere.

    python tests/golden/make_reference_shape_bounds_vectors.py

Sets: w4 / w8 / w16 (random worlds with hull bundle width 4, 8, 16: every type, compounds with hull children, big compounds, meshes of a few
hundred triangles with non-uniform scale, slow and fast spins) and zero (the signed-zero fixture: flat hulls and flat meshes whose points sit on
z = +-0, at position (-0, -0, -0) with -0 velocity components, so that the sign of the winning zero reaches the output's max.z).
Per set: the library arrays (lib_*), per body shape / margins / allow / q / pos / lin / ang (velocity after the callback), dt, out[n, 7]."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle", "ref_transpile"))
import shape_bounds_ref  # noqa: E402

from bepuphysics2_b200 import scenes  # noqa: E402
from bepuphysics2_b200.native import ShapeLibrary, typed_index  # noqa: E402

FP = C.POINTER(C.c_float)
LIBRARY_FIELDS = ("spheres", "capsules", "boxes", "triangles", "cylinders", "hull_points", "hulls", "compound_children", "compounds", "big_compounds", "mesh_triangles", "meshes")


def random_set(width, seed, bodies=160):
    rng = np.random.default_rng(seed)
    library = scenes.shape_library(rng, hull_width=width, primitives=16, hulls=12, hull_points=(5, 64), compounds=10, big_compounds=4, compound_children=(1, 24),
                                   mesh_triangle_counts=(200, 350))
    world = scenes.shape_world(bodies, seed=seed + 1, library=library, type_weights={0: 1, 1: 1, 2: 1, 3: 2, 4: 1, 5: 3, 6: 3, 7: 2, 8: 1, "none": 0.2, "user": 0.2})
    b = world["bodies"]
    c = world["collidables"]
    return library, c["shape"], np.stack([c["minimum_speculative_margin"], c["maximum_speculative_margin"]], axis=1), c["allow_expansion_beyond_speculative_margin"], \
        b[:, 0:4].copy(), b[:, 4:7].copy(), b[:, 8:11].copy(), b[:, 12:15].copy()


def signed_zero_set(width, seed):
    """Flat hulls and flat meshes on z = +-0 (x, y < 0 so that the rotation by the identity keeps the sign of z), identity orientation, position and
    velocity all -0, zero minimum margin: max.z of the output is the sign of the zero the fold kept."""
    rng = np.random.default_rng(seed)
    hulls, bundles, first = [], [], 0
    for _ in range(8):
        n = int(rng.integers(width + 1, 4 * width))
        pts = np.stack([-rng.uniform(0.5, 2, n), -rng.uniform(0.5, 2, n), np.where(rng.random(n) < 0.5, -0.0, 0.0)], axis=1).astype(np.float32)
        bb = scenes.bundle_hull_points(pts, width)
        bundles.append(bb)
        hulls.append((first, bb.shape[0]))
        first += bb.shape[0]
    mesh_pool, meshes = [], []
    for _ in range(4):
        n = int(rng.integers(3, 40))
        tri = np.zeros((n, 3, 3), dtype=np.float32)
        tri[:, :, 0] = -rng.uniform(0.5, 2, (n, 3))
        tri[:, :, 1] = -rng.uniform(0.5, 2, (n, 3))
        tri[:, :, 2] = np.where(rng.random((n, 3)) < 0.5, -0.0, 0.0)
        meshes.append((sum(len(m) for m in mesh_pool), n, (1.5, 0.5, 2.0)))
        mesh_pool.append(tri.reshape(n, 9))
    library = ShapeLibrary(spheres=[1.0], hull_points=np.concatenate(bundles), hull_bundle_width=width, hulls=hulls, mesh_triangles=np.concatenate(mesh_pool), meshes=meshes)
    shapes = np.concatenate([typed_index(np.full(8, 5), np.arange(8)), typed_index(np.full(4, 8), np.arange(4))])
    n = shapes.shape[0]
    margins = np.tile(np.array([[0.0, 3.40282347e+38]], dtype=np.float32), (n, 1))
    q = np.tile(np.array([[0, 0, 0, 1]], dtype=np.float32), (n, 1))
    negzero = np.full((n, 3), -0.0, dtype=np.float32)
    return library, shapes, margins, np.zeros(n, dtype=np.int32), q, negzero.copy(), negzero.copy(), negzero.copy()


def evaluate(lib, library, shapes, margins, allow, q, pos, lin, ang, dt):
    desc = library.desc()
    out = np.zeros((shapes.shape[0], 7), dtype=np.float32)
    for i in range(shapes.shape[0]):
        rc = lib.ref_shape_bounds(C.addressof(desc), int(shapes[i]), margins[i].ctypes.data_as(FP), int(allow[i]), q[i].ctypes.data_as(FP), pos[i].ctypes.data_as(FP),
                                  lin[i].ctypes.data_as(FP), ang[i].ctypes.data_as(FP), dt, out[i].ctypes.data_as(FP))
        if rc != 0:
            out[i] = 0.0  # no shape / user-registered type: no built-in bounds
    return out


def main():
    lib = C.CDLL(shape_bounds_ref.build())
    lib.ref_shape_bounds.argtypes = [C.c_void_p, C.c_uint32, FP, C.c_int32, FP, FP, FP, FP, C.c_float, FP]
    out = {}
    sets = [("w4", random_set(4, 41), 1.0 / 60.0), ("w8", random_set(8, 42), 1.0 / 60.0), ("w16", random_set(16, 43), 1.0 / 240.0), ("zero", signed_zero_set(8, 44), 1.0 / 60.0)]
    for name, (library, *inputs), dt in sets:
        for f in LIBRARY_FIELDS:
            out["%s_lib_%s" % (name, f)] = getattr(library, f)
        out["%s_width" % name] = np.int32(library.hull_bundle_width)
        for field, a in zip(("shape", "margins", "allow", "q", "pos", "lin", "ang"), inputs):
            out["%s_%s" % (name, field)] = np.ascontiguousarray(a)
        out["%s_dt" % name] = np.float32(dt)
        out["%s_out" % name] = evaluate(lib, library, *[np.ascontiguousarray(a) for a in inputs], dt)
    path = os.path.join(ROOT, "tests", "golden", "reference_shape_bounds_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, {k: v.shape for k, v in out.items() if k.endswith("_out")})


if __name__ == "__main__":
    main()
