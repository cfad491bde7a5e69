// Per-element arithmetic of PredictBoundingBoxes for every built-in shape type (see bepu_shape_bounds.cu): triangles, convex hulls, compounds, big
// compounds and meshes, on top of the convex-primitive arithmetic of bepu_bounds_math.cuh. Plain scalar fp32 behind __device__, in its own header so
// that tests/device_on_host can compile it for the host and hold it to the reference-derived vectors without a GPU. Expression shapes follow the
// reference (file:line per function); compiled without FMA contraction.
//
// The reductions the kernels run in parallel (hull lanes, compound children, mesh triangles) are written here as their sequential steps; each step
// states which operand survives a tie, because Vector.Min / Vector3.Min are (a < b) ? a : b and -0 == +0: the order of a fold decides the sign of
// a zero extreme.
#pragma once
#include <string.h>

#include "bepu_bounds_math.cuh"

namespace BEPU_NS {

// Records in the layouts of include/bepucuda.h (which are the reference's own where it has a flat layout).
struct HullRecord { int32_t first_bundle, bundle_count; };
struct CompoundRecord { int32_t first_child, child_count; };
struct CompoundChildRecord { float local_orientation[4]; float local_position[3]; uint32_t shape; };  // Compound.cs:L18-31
struct MeshRecord { int64_t first_triangle; int32_t triangle_count; float scale[3]; };
struct BodyCollidableRecord { uint32_t shape; float minimum_speculative_margin, maximum_speculative_margin; int32_t allow_expansion_beyond_speculative_margin; };

// The shape library as the kernels see it: one pointer per reference shape batch (Sphere {Radius}, Capsule {Radius, HalfLength}, Box {HalfWidth,
// HalfHeight, HalfLength}, Triangle {A, B, C}, Cylinder {Radius, HalfLength}), the hull point bundles (Vector3Wide of width hull_width, AOSOA),
// the compound child pool and the mesh triangle pool.
struct ShapeLibraryView {
    const float *spheres, *capsules, *boxes, *triangles, *cylinders, *hull_points;
    const HullRecord* hulls;
    const CompoundChildRecord* compound_children;
    const CompoundRecord *compounds, *big_compounds;
    const float* mesh_triangles;
    const MeshRecord* meshes;
    int32_t hull_width;
};

enum : int32_t { kSphere = 0, kCapsule = 1, kBox = 2, kTriangle = 3, kCylinder = 4, kConvexHull = 5, kCompound = 6, kBigCompound = 7, kMesh = 8 };

// TypedIndex (TypedIndex.cs:L23-51)
BEPU_DI bool typed_index_exists(uint32_t packed) { return (packed & 0x80000000u) != 0u; }
BEPU_DI int32_t typed_index_type(uint32_t packed) { return (int32_t)((packed & 0x7F000000u) >> 24); }
BEPU_DI int32_t typed_index_index(uint32_t packed) { return (int32_t)(packed & 0x00FFFFFFu); }

BEPU_DI uint32_t float_bits(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    return u;
}
// MathF.Max / MathF.Min (System.Math, .NET 8): IEEE 754:2019 maximum / minimum, NaN-propagating, +0 > -0. Not the Vector.Max lane rule.
BEPU_DI float mathf_max(float x, float y) {
    if (x != y) return x == x ? (y < x ? x : y) : x;
    return (float_bits(y) >> 31) ? x : y;
}
BEPU_DI float mathf_min(float x, float y) {
    if (x != y) return x == x ? (x < y ? x : y) : x;
    return (float_bits(x) >> 31) ? x : y;
}

// ---- narrow System.Numerics / BepuUtilities helpers (restated apart from the wide ones in bepu_device_math.cuh) ------------------------------
BEPU_DI V3 vmin3(V3 a, V3 b) { return {a.x < b.x ? a.x : b.x, a.y < b.y ? a.y : b.y, a.z < b.z ? a.z : b.z}; }  // Vector3.Min: ties -> b
BEPU_DI V3 vmax3(V3 a, V3 b) { return {a.x > b.x ? a.x : b.x, a.y > b.y ? a.y : b.y, a.z > b.z ? a.z : b.z}; }  // Vector3.Max: ties -> b
BEPU_DI V3 vabs3(V3 a) { return {fabsf(a.x), fabsf(a.y), fabsf(a.z)}; }
BEPU_DI V3 vmul3(V3 a, V3 b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
BEPU_DI float narrow_length_squared(V3 v) { return v.x * v.x + v.y * v.y + v.z * v.z; }  // Vector3.LengthSquared = Dot(v, v)
BEPU_DI float narrow_length(V3 v) { return sqrtf(narrow_length_squared(v)); }

// Matrix3x3.CreateFromQuaternion (BepuUtilities/Matrix3x3.cs:L306-335)
BEPU_DI M33 narrow_matrix_from_quaternion(Q4 q) {
    const float qX2 = q.x + q.x, qY2 = q.y + q.y, qZ2 = q.z + q.z;
    const float XX = qX2 * q.x, YY = qY2 * q.y, ZZ = qZ2 * q.z;
    const float XY = qX2 * q.y, XZ = qX2 * q.z, XW = qX2 * q.w;
    const float YZ = qY2 * q.z, YW = qY2 * q.w, ZW = qZ2 * q.w;
    M33 r;
    r.x = {1.0f - YY - ZZ, XY + ZW, XZ - YW};
    r.y = {XY - ZW, 1.0f - XX - ZZ, YZ + XW};
    r.z = {XZ + YW, YZ - XW, 1.0f - XX - YY};
    return r;
}
// Matrix3x3.Transform (Matrix3x3.cs:L200-206): m.X * broadcast(v.X) + m.Y * broadcast(v.Y) + m.Z * broadcast(v.Z)
BEPU_DI V3 narrow_transform(V3 v, const M33& m) {
    return {m.x.x * v.x + m.y.x * v.y + m.z.x * v.z, m.x.y * v.x + m.y.y * v.y + m.z.y * v.z, m.x.z * v.x + m.y.z * v.y + m.z.z * v.z};
}
// QuaternionEx.ConcatenateWithoutOverlap (BepuUtilities/QuaternionEx.cs:L50-56)
BEPU_DI Q4 narrow_concatenate(Q4 a, Q4 b) {
    return {a.w * b.x + a.x * b.w + a.z * b.y - a.y * b.z, a.w * b.y + a.y * b.w + a.x * b.z - a.z * b.x, a.w * b.z + a.z * b.w + a.y * b.x - a.x * b.y,
            a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
// QuaternionEx.TransformWithoutOverlap (QuaternionEx.cs:L373-395), reached through QuaternionEx.Transform (L405-409)
BEPU_DI V3 narrow_transform(V3 v, Q4 r) {
    const float x2 = r.x + r.x, y2 = r.y + r.y, z2 = r.z + r.z;
    const float xx2 = r.x * x2, xy2 = r.x * y2, xz2 = r.x * z2, yy2 = r.y * y2, yz2 = r.y * z2, zz2 = r.z * z2;
    const float wx2 = r.w * x2, wy2 = r.w * y2, wz2 = r.w * z2;
    return {v.x * (1.0f - yy2 - zz2) + v.y * (xy2 - wz2) + v.z * (xz2 + wy2), v.x * (xy2 + wz2) + v.y * (1.0f - xx2 - zz2) + v.z * (yz2 - wx2),
            v.x * (xz2 - wy2) + v.y * (yz2 + wx2) + v.z * (1.0f - xx2 - yy2)};
}

// Local bounds of a convex shape: min, max, maximumRadius, maximumAngularExpansion (IConvexShape wide GetBounds, one lane).
struct ConvexLocalBounds { V3 min, max; float maximumRadius, maximumAngularExpansion; };

// TriangleWide.GetBounds (Collidables/Triangle.cs:L203-221)
BEPU_DI ConvexLocalBounds triangle_bounds(const float* t, Q4 orientation) {
    const V3 A = {t[0], t[1], t[2]}, B = {t[3], t[4], t[5]}, C = {t[6], t[7], t[8]};
    const M33 basis = matrix_from_quaternion(orientation);  // Matrix3x3Wide.CreateFromQuaternion
    const V3 worldA = transform(A, basis), worldB = transform(B, basis), worldC = transform(C, basis);  // Matrix3x3Wide.TransformWithoutOverlap
    ConvexLocalBounds r;
    r.min = {fmin_ps(worldA.x, fmin_ps(worldB.x, worldC.x)), fmin_ps(worldA.y, fmin_ps(worldB.y, worldC.y)), fmin_ps(worldA.z, fmin_ps(worldB.z, worldC.z))};
    r.max = {fmax_ps(worldA.x, fmax_ps(worldB.x, worldC.x)), fmax_ps(worldA.y, fmax_ps(worldB.y, worldC.y)), fmax_ps(worldA.z, fmax_ps(worldB.z, worldC.z))};
    const float aLengthSquared = length_squared(A), bLengthSquared = length_squared(B), cLengthSquared = length_squared(C);
    r.maximumRadius = sqrtf(fmax_ps(aLengthSquared, fmax_ps(bLengthSquared, cLengthSquared)));
    r.maximumAngularExpansion = r.maximumRadius;
    return r;
}

// ---- ConvexHullWide.GetBounds (ConvexHull.cs:L319-364) ----------------------------------------------------------------------------------
// Lane `slot` of the reference's loop over the hull's point bundles: min / max / max |p|^2 folded over the bundles in order. Vector3Wide.Min(minWide, p)
// keeps p on a tie, so the LATER bundle wins within a lane.
struct HullLane { V3 min, max; float maximumRadiusSquared; };
BEPU_DI HullLane hull_lane_fold(const float* hullPoints, int32_t width, HullRecord hull, int32_t slot, const M33& orientationMatrix) {
    HullLane r = {{3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f}, {-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f}, 0.0f};
    for (int32_t j = 0; j < hull.bundle_count; ++j) {
        const float* bundle = hullPoints + ((size_t)hull.first_bundle + (size_t)j) * 3 * (size_t)width;
        const V3 localPoint = {bundle[slot], bundle[width + slot], bundle[2 * width + slot]};
        const V3 p = transform(localPoint, orientationMatrix);  // Matrix3x3Wide.TransformWithoutOverlap
        const float lengthSquared = length_squared(localPoint);  // Vector3Wide.LengthSquared
        r.maximumRadiusSquared = fmax_ps(lengthSquared, r.maximumRadiusSquared);
        r.min = {fmin_ps(r.min.x, p.x), fmin_ps(r.min.y, p.y), fmin_ps(r.min.z, p.z)};
        r.max = {fmax_ps(r.max.x, p.x), fmax_ps(r.max.y, p.y), fmax_ps(r.max.z, p.z)};
    }
    return r;
}
// The horizontal step over the lanes (ConvexHull.cs:L341-351): Vector3.Min(candidate, running) keeps `running` on a tie, so the LOWER lane wins.
BEPU_DI void hull_lane_merge(HullLane& running, const HullLane& candidate) {
    running.min = vmin3(candidate.min, running.min);
    running.max = vmax3(candidate.max, running.max);
    if (candidate.maximumRadiusSquared > running.maximumRadiusSquared) running.maximumRadiusSquared = candidate.maximumRadiusSquared;
}
BEPU_DI ConvexLocalBounds hull_finish(const HullLane& folded) {
    ConvexLocalBounds r;
    r.min = folded.min;
    r.max = folded.max;
    r.maximumRadius = sqrtf(folded.maximumRadiusSquared);  // the radius of the LOCAL points
    r.maximumAngularExpansion = r.maximumRadius;
    return r;
}
// The whole hull in one thread, lanes in order (a compound's hull child).
BEPU_DI ConvexLocalBounds hull_bounds(const float* hullPoints, int32_t width, HullRecord hull, Q4 orientation) {
    const M33 orientationMatrix = matrix_from_quaternion(orientation);  // Matrix3x3Wide.CreateFromQuaternion of the rebroadcast orientation
    HullLane running = hull_lane_fold(hullPoints, width, hull, 0, orientationMatrix);
    for (int32_t slot = 1; slot < width; ++slot) hull_lane_merge(running, hull_lane_fold(hullPoints, width, hull, slot, orientationMatrix));
    return hull_finish(running);
}

// Local bounds of a convex shape of type 0-5 from the library (ExecuteConvexBatch's shapeWide.GetBounds).
BEPU_DI ConvexLocalBounds convex_local_bounds(const ShapeLibraryView& lib, int32_t type, int32_t index, Q4 orientation) {
    if (type == kTriangle) return triangle_bounds(lib.triangles + 9 * (size_t)index, orientation);
    if (type == kConvexHull) return hull_bounds(lib.hull_points, lib.hull_width, lib.hulls[index], orientation);
    ConvexShape s = {type, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0};
    if (type == kSphere) {
        s.a = lib.spheres[index];
    } else if (type == kBox) {
        s.a = lib.boxes[3 * (size_t)index], s.b = lib.boxes[3 * (size_t)index + 1], s.c = lib.boxes[3 * (size_t)index + 2];
    } else {
        const float* d = (type == kCapsule ? lib.capsules : lib.cylinders) + 2 * (size_t)index;
        s.a = d[0], s.b = d[1];
    }
    const LocalBounds local = shape_bounds(s, orientation);
    return {-local.max, local.max, local.maximumRadius, local.maximumAngularExpansion};
}

BEPU_DI void expand_convex_bounds(const ConvexLocalBounds& local, const BodyCollidableRecord& c, V3 position, const Velocity& velocity, float dt, V3& bundleMin, V3& bundleMax,
                                  float& speculativeMargin) {
    expand_convex_bounds(local.min, local.max, local.maximumRadius, local.maximumAngularExpansion, c.minimum_speculative_margin, c.maximum_speculative_margin,
                         c.allow_expansion_beyond_speculative_margin, position, velocity, dt, bundleMin, bundleMax, speculativeMargin);
}

// ---- compounds: Compound.AddChildBoundsToBatcher (Compound.cs:L198-221) + ExecuteConvexBatch's CompoundChild merge (BoundingBoxBatcher.cs:L208-214)
struct MergedBounds { V3 min, max; float speculativeMargin; };
// ExecuteCompoundBatch (BoundingBoxBatcher.cs:L268-287): margin 0, box (+MaxValue, -MaxValue) before the first child.
BEPU_DI MergedBounds merged_bounds_start() { return {{3.40282347e+38f, 3.40282347e+38f, 3.40282347e+38f}, {-3.40282347e+38f, -3.40282347e+38f, -3.40282347e+38f}, 0.0f}; }
// One merge: MathF.Max of the margins, BoundingBox.CreateMerged (BepuUtilities/BoundingBox.cs:L173-177: Vector3.Min(running, child)), so the
// LATER child wins a tie.
BEPU_DI void merge_bounds(MergedBounds& running, const MergedBounds& later) {
    running.speculativeMargin = mathf_max(running.speculativeMargin, later.speculativeMargin);
    running.min = vmin3(running.min, later.min);
    running.max = vmax3(running.max, later.max);
}
// The bounds ExecuteConvexBatch produces for one child of a compound body.
BEPU_DI MergedBounds compound_child_bounds(const ShapeLibraryView& lib, const CompoundChildRecord& child, const BodyCollidableRecord& parent, Q4 orientation, V3 position,
                                           const Velocity& velocity, float dt) {
    // Compound.GetRotatedChildPose (Compound.cs:L153-157)
    const Q4 localOrientation = {child.local_orientation[0], child.local_orientation[1], child.local_orientation[2], child.local_orientation[3]};
    const Q4 childOrientation = narrow_concatenate(localOrientation, orientation);
    V3 childPosition = narrow_transform(V3{child.local_position[0], child.local_position[1], child.local_position[2]}, orientation);
    V3 angularContributionToChildLinear = cross(velocity.ang, childPosition);
    const float contributionLengthSquared = narrow_length_squared(angularContributionToChildLinear);
    const float localPoseRadiusSquared = narrow_length_squared(childPosition);
    if (contributionLengthSquared > localPoseRadiusSquared) {
        // (float)(Math.Sqrt(localPoseRadiusSquared) / Math.Sqrt(contributionLengthSquared)): double sqrt and division, then one rounding to float
        angularContributionToChildLinear = angularContributionToChildLinear * (float)(sqrt((double)localPoseRadiusSquared) / sqrt((double)contributionLengthSquared));
    }
    const Velocity childVelocity = {velocity.lin + angularContributionToChildLinear, velocity.ang};
    childPosition = childPosition + position;
    const ConvexLocalBounds local = convex_local_bounds(lib, typed_index_type(child.shape), typed_index_index(child.shape), childOrientation);
    MergedBounds r;
    expand_convex_bounds(local, parent, childPosition, childVelocity, dt, r.min, r.max, r.speculativeMargin);
    return r;
}

// ---- meshes: Mesh.ComputeBounds (Mesh.cs:L232-255) + ExecuteHomogeneousCompoundBatch (BoundingBoxBatcher.cs:L225-266) -------------------------
// The triangle's vertices, scaled and rotated: Matrix3x3.Transform(scale * vertex, r).
BEPU_DI void mesh_triangle_vertices(const float* t, V3 scale, const M33& r, V3& a, V3& b, V3& c) {
    a = narrow_transform(vmul3(scale, V3{t[0], t[1], t[2]}), r);
    b = narrow_transform(vmul3(scale, V3{t[3], t[4], t[5]}), r);
    c = narrow_transform(vmul3(scale, V3{t[6], t[7], t[8]}), r);
}
// One step of the mesh's sequential min / max fold, per coordinate, with the position of the surviving value:
//   min0 = Min(a, b); min1 = Min(c, min); min = Min(min0, min1)
// so on a tie the running value survives (the FIRST triangle that reaches an extreme wins) and within that triangle c beats b beats a. `key` is the
// index of the triangle the running value came from; a parallel reduction over (value, key) with "smaller key wins a tie" then reproduces the fold.
BEPU_DI void mesh_fold_min(float a, float b, float c, int32_t triangle, float& running, int32_t& key) {
    const float min0 = a < b ? a : b;
    const float min1 = c < running ? c : running;
    const bool keep = !(min0 < min1) && !(c < running);
    running = min0 < min1 ? min0 : min1;
    key = keep ? key : triangle;
}
BEPU_DI void mesh_fold_max(float a, float b, float c, int32_t triangle, float& running, int32_t& key) {
    const float max0 = a > b ? a : b;
    const float max1 = c > running ? c : running;
    const bool keep = !(max0 > max1) && !(c > running);
    running = max0 > max1 ? max0 : max1;
    key = keep ? key : triangle;
}
// Combining two partial folds over disjoint triangle sets: the smaller value, on a tie the smaller key (the earlier triangle).
BEPU_DI void mesh_combine_min(float& value, int32_t& key, float otherValue, int32_t otherKey) {
    if (otherValue < value || (!(value < otherValue) && otherKey < key)) value = otherValue, key = otherKey;
}
BEPU_DI void mesh_combine_max(float& value, int32_t& key, float otherValue, int32_t otherKey) {
    if (otherValue > value || (!(value > otherValue) && otherKey < key)) value = otherValue, key = otherKey;
}

// BoundingBoxHelpers.GetAngularBoundsExpansion, scalar overload (BoundingBoxHelpers.cs:L125-133): (float)Math.Sqrt of the float product.
BEPU_DI float narrow_angular_bounds_expansion(float angularVelocityMagnitude, float dt, float maximumRadius, float maximumAngularExpansion) {
    const float a = fmin_ps(angularVelocityMagnitude * dt, 3.14159274f / 3.0f);  // MathHelper.Min
    const float a2 = a * a;
    const float a4 = a2 * a2;
    const float a6 = a4 * a2;
    const float cosAngleMinusOne = a2 * (-1.0f / 2.0f) + a4 * (1.0f / 24.0f) - a6 * (1.0f / 720.0f);
    return fmin_ps(maximumAngularExpansion, (float)sqrt((double)(-2.0f * maximumRadius * maximumRadius * cosAngleMinusOne)));
}
// ExecuteHomogeneousCompoundBatch from the mesh's rotated (min, max) onwards (BoundingBoxBatcher.cs:L243-264), narrow Vector3 arithmetic throughout.
BEPU_DI void mesh_bounds(V3 min, V3 max, const BodyCollidableRecord& c, V3 position, const Velocity& velocity, float dt, V3& boundsMin, V3& boundsMax, float& speculativeMargin) {
    const V3 absMin = vabs3(min), absMax = vabs3(max);
    const float maximumRadius = narrow_length(vmax3(absMin, absMax));
    const V3 minimumComponents = vmin3(absMin, absMax);
    const float minimumRadius = fmin_ps(minimumComponents.x, fmin_ps(minimumComponents.y, minimumComponents.z));  // MathHelper.Min
    const float maximumAngularExpansion = maximumRadius - minimumRadius;
    const float angularBoundsExpansion = narrow_angular_bounds_expansion(narrow_length(velocity.ang), dt, maximumRadius, maximumAngularExpansion);
    speculativeMargin = narrow_length(velocity.lin) * dt + angularBoundsExpansion;
    speculativeMargin = mathf_max(c.minimum_speculative_margin, mathf_min(c.maximum_speculative_margin, speculativeMargin));
    const float maximumAllowedExpansion = c.allow_expansion_beyond_speculative_margin ? 3.40282347e+38f : speculativeMargin;
    // BoundingBoxHelpers.GetBoundsExpansion, Vector3 overload (BoundingBoxHelpers.cs:L142-149)
    const V3 linearDisplacement = velocity.lin * dt;
    const V3 zero = {0.0f, 0.0f, 0.0f}, broadcastExpansion = {angularBoundsExpansion, angularBoundsExpansion, angularBoundsExpansion};
    V3 minExpansion = vmin3(zero, linearDisplacement) - broadcastExpansion;
    V3 maxExpansion = vmax3(zero, linearDisplacement) + broadcastExpansion;
    const V3 broadcastMaximumBoundsExpansion = {maximumAllowedExpansion, maximumAllowedExpansion, maximumAllowedExpansion};
    minExpansion = vmax3(-broadcastMaximumBoundsExpansion, minExpansion);
    maxExpansion = vmin3(broadcastMaximumBoundsExpansion, maxExpansion);
    boundsMin = position + (min + minExpansion);
    boundsMax = position + (max + maxExpansion);
}

}  // namespace BEPU_NS
