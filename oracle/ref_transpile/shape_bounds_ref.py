"""ORACLE PINNING — test infrastructure only. Recipe for oracle/_ref/libbepu_ref_shapes.so: the reference's C# for PredictBoundingBoxes over every
built-in shape type, transpiled mechanically by cs2cpp.py's Transpiler (used as a library, unchanged) with a wider source list, and compiled with
shape_bounds_harness.cpp (the glue for the loops the transpiler cannot carry) with g++ -ffp-contract=off.

On top of cs2cpp's own sources it takes TriangleWide.GetBounds and the narrow helpers compound children and meshes go through:
QuaternionEx.ConcatenateWithoutOverlap / TransformWithoutOverlap, Matrix3x3.CreateFromQuaternion / Transform and the Vector3 overloads of
BoundingBoxHelpers. Members that use the narrow System.Numerics types Vector3 / Quaternion / Matrix3x3 are admitted for those types only; their lane
semantics come from ref_runtime_narrow.h. Outputs go to oracle/_ref/ only (git-ignored). build() returns None where the reference tree is absent
and no prebuilt library exists.

    python oracle/ref_transpile/shape_bounds_ref.py            # build (tests/golden/make_reference_shape_bounds_vectors.py calls build())
"""
import os
import re
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "_ref")
LIB = os.path.join(OUT, "libbepu_ref_shapes.so")
REFERENCE = os.environ.get("BEPU_REFERENCE_ROOT", "/root/reference")

EXTRA_SOURCES = [("BepuPhysics/Collidables/Triangle.cs", ["TriangleWide"]), ("BepuUtilities/QuaternionEx.cs", ["QuaternionEx"]), ("BepuUtilities/Matrix3x3.cs", ["Matrix3x3"])]
EXTRA_ONLY_METHODS = {"TriangleWide": {"GetBounds"}, "QuaternionEx": {"ConcatenateWithoutOverlap", "TransformWithoutOverlap"}, "Matrix3x3": {"CreateFromQuaternion", "Transform"}}
# Types whose named members may use these narrow types (every other member that names a narrow type stays skipped, as in cs2cpp).
NARROW_OK = {"BoundingBoxHelpers", "QuaternionEx", "Matrix3x3"}
NARROW_CARRIED = {"Vector3", "Quaternion", "Matrix3x3"}


def transpile(header):
    sys.path.insert(0, HERE)
    import cs2cpp

    cs2cpp.SOURCES = cs2cpp.SOURCES + EXTRA_SOURCES
    cs2cpp.ONLY_METHODS = dict(cs2cpp.ONLY_METHODS, **EXTRA_ONLY_METHODS)
    narrow = frozenset(cs2cpp.NARROW)
    current = [None]

    class NarrowFilter:
        """Stands in for cs2cpp.NARROW: `words & NARROW` in parse_type drops a member that names a narrow type, except for the narrow types
        ref_runtime_narrow.h carries when the member belongs to a NARROW_OK type."""

        def __rand__(self, words):
            hit = set(words) & narrow
            return set() if current[0] in NARROW_OK and hit <= NARROW_CARRIED else hit

        def __contains__(self, name):
            return name in narrow

    cs2cpp.NARROW = NarrowFilter()
    parse_type = cs2cpp.parse_type

    def parse_type_tracking(kind, name, generic, body):
        current[0] = name
        return parse_type(kind, name, generic, body)

    cs2cpp.parse_type = parse_type_tracking

    class Transpiler(cs2cpp.Transpiler):
        def translate_expr(self, owner, body):
            body = super().translate_expr(owner, body)
            body = re.sub(r"(?<![\w.:])Vector3\.(?=\w)", "Vector3::", body)  # static members of System.Numerics.Vector3
            return re.sub(r"\bVector3::Zero\b(?!\s*\()", "Vector3::Zero()", body)

    tr = Transpiler(REFERENCE)
    tr.load()
    text, skipped = tr.emit()
    text = text.replace('#include "ref_runtime.h"', '#include "ref_runtime_narrow.h"', 1)
    with open(header, "w") as f:
        f.write(text)
    for s in skipped:
        print("note:", s, file=sys.stderr)


def build(force=False):
    have_reference = os.path.isdir(os.path.join(REFERENCE, "BepuPhysics", "Collidables"))
    sources = [os.path.join(HERE, f) for f in ("cs2cpp.py", "ref_runtime.h", "ref_runtime_narrow.h", "shape_bounds_ref.py", "shape_bounds_harness.cpp")]
    if os.path.exists(LIB) and not force and (not have_reference or all(os.path.getmtime(s) <= os.path.getmtime(LIB) for s in sources)):
        return LIB
    if not have_reference:
        return None
    os.makedirs(OUT, exist_ok=True)
    for f in ("ref_runtime.h", "ref_runtime_narrow.h", "shape_bounds_harness.cpp"):
        shutil.copy(os.path.join(HERE, f), os.path.join(OUT, f))
    header = os.path.join(OUT, "bepu_ref_shapes_generated.h")
    # in a process of its own: transpile() rebinds module globals of cs2cpp
    subprocess.check_call([sys.executable, os.path.abspath(__file__), "--transpile", header])
    subprocess.check_call(["/usr/bin/g++", "-O1", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-march=x86-64-v3", "-shared", "-o", LIB,
                           os.path.join(OUT, "shape_bounds_harness.cpp")])
    return LIB


if __name__ == "__main__":
    if "--transpile" in sys.argv:
        transpile(sys.argv[sys.argv.index("--transpile") + 1])
    else:
        print(build(force="--force" in sys.argv))
