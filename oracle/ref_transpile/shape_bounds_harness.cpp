// ORACLE PINNING — test infrastructure only. Harness of oracle/_ref/libbepu_ref_shapes.so (oracle/ref_transpile/shape_bounds_ref.py): PredictBoundingBoxes
// for every built-in shape type over the reference's own C# text, transpiled into bepu_ref_shapes_generated.h (TriangleWide / CapsuleWide / BoxWide /
// CylinderWide.GetBounds, BoundingBoxHelpers, Matrix3x3Wide, Vector3Wide, QuaternionEx.ConcatenateWithoutOverlap / TransformWithoutOverlap,
// Matrix3x3.CreateFromQuaternion / Transform). What the transpiler cannot carry is written here as glue over those calls, each part citing the C# it
// follows: the ExecuteConvexBatch body, ConvexHullWide.GetBounds' walk over its point Buffer, the compound child loop with the batcher's merge, the
// mesh triangle loop and ExecuteHomogeneousCompoundBatch. Compiled -ffp-contract=off.
#include "bepu_ref_shapes_generated.h"

#include <cstring>

using namespace bepu_ref;

static QuaternionWide quat(const float* f) { QuaternionWide q; q.X = f[0]; q.Y = f[1]; q.Z = f[2]; q.W = f[3]; return q; }
static Vector3Wide vec3(const float* f) { Vector3Wide v; v.X = f[0]; v.Y = f[1]; v.Z = f[2]; return v; }

// Convex-primitive bounds of PredictBoundingBoxes: transpiled CapsuleWide / BoxWide / CylinderWide / TriangleWide.GetBounds and BoundingBoxHelpers.GetAngularBoundsExpansion /
// GetBoundsExpansion, glued exactly like BoundingBoxBatcher.ExecuteConvexBatch (Collidables/BoundingBoxBatcher.cs:L176-197) glues them. SphereWide.GetBounds
// (Sphere.cs:L149-160: max = radius, min = -radius, no angular expansion) is three assignments and is written out here (its `new Vector3Wide(ref x)` overload pair has no C++ counterpart).
static void ref_convex_local(int type, const float* dims, QuaternionWide orientations, Vector<float>& maximumRadius, Vector<float>& maximumAngularExpansion, Vector3Wide& bundleMin, Vector3Wide& bundleMax) {
    if (type == 0) { maximumRadius = Vector<float>(0.0f); maximumAngularExpansion = Vector<float>(0.0f); Vector<float> Radius(dims[0]); Vector<float> negatedRadius = -Radius;
        bundleMax.X = Radius; bundleMax.Y = Radius; bundleMax.Z = Radius; bundleMin.X = negatedRadius; bundleMin.Y = negatedRadius; bundleMin.Z = negatedRadius; }
    else if (type == 1) { CapsuleWide s; s.Radius = dims[0]; s.HalfLength = dims[1]; s.GetBounds(orientations, 1, maximumRadius, maximumAngularExpansion, bundleMin, bundleMax); }
    else if (type == 2) { BoxWide s; s.HalfWidth = dims[0]; s.HalfHeight = dims[1]; s.HalfLength = dims[2]; s.GetBounds(orientations, 1, maximumRadius, maximumAngularExpansion, bundleMin, bundleMax); }
    else if (type == 3) { TriangleWide s; s.A = vec3(dims); s.B = vec3(dims + 3); s.C = vec3(dims + 6); s.GetBounds(orientations, 1, maximumRadius, maximumAngularExpansion, bundleMin, bundleMax); }
    else { CylinderWide s; s.Radius = dims[0]; s.HalfLength = dims[1]; s.GetBounds(orientations, 1, maximumRadius, maximumAngularExpansion, bundleMin, bundleMax); }
}
// ExecuteConvexBatch from the shape's bounds onwards (BoundingBoxBatcher.cs:L181-197). out: min.xyz, margin, max.xyz.
static void ref_convex_expand(Vector<float> maximumRadius, Vector<float> maximumAngularExpansion, Vector3Wide bundleMin, Vector3Wide bundleMax, const float* margins, int allow, const float* pos,
                              const float* lin, const float* ang, float dt, float* out) {
    Vector3Wide positions = vec3(pos); BodyVelocityWide velocities; velocities.Linear = vec3(lin); velocities.Angular = vec3(ang); Vector<float> dtWide(dt);
    Vector<float> angularSpeed; Vector3Wide::Length(velocities.Angular, angularSpeed); Vector<float> linearSpeed; Vector3Wide::Length(velocities.Linear, linearSpeed);
    auto angularBoundsExpansion = BoundingBoxHelpers::GetAngularBoundsExpansion(angularSpeed, dtWide, maximumRadius, maximumAngularExpansion);
    auto speculativeMargin = linearSpeed * dtWide + angularBoundsExpansion;
    speculativeMargin = VectorOps::Max(Vector<float>(margins[0]), VectorOps::Min(Vector<float>(margins[1]), speculativeMargin));
    auto maximumBoundsExpansion = VectorOps::ConditionalSelect(Vector<int>(allow ? -1 : 0), Vector<float>(3.40282347e+38f), speculativeMargin);
    Vector3Wide minExpansion, maxExpansion; BoundingBoxHelpers::GetBoundsExpansion(velocities.Linear, dtWide, angularBoundsExpansion, minExpansion, maxExpansion);
    Vector3Wide negated; negated.X = -maximumBoundsExpansion; negated.Y = -maximumBoundsExpansion; negated.Z = -maximumBoundsExpansion;
    minExpansion.X = VectorOps::Max(negated.X, minExpansion.X); minExpansion.Y = VectorOps::Max(negated.Y, minExpansion.Y); minExpansion.Z = VectorOps::Max(negated.Z, minExpansion.Z);
    maxExpansion.X = VectorOps::Min(maximumBoundsExpansion, maxExpansion.X); maxExpansion.Y = VectorOps::Min(maximumBoundsExpansion, maxExpansion.Y); maxExpansion.Z = VectorOps::Min(maximumBoundsExpansion, maxExpansion.Z);
    bundleMin = positions + (bundleMin + minExpansion); bundleMax = positions + (bundleMax + maxExpansion);
    out[0] = bundleMin.X.v; out[1] = bundleMin.Y.v; out[2] = bundleMin.Z.v; out[3] = speculativeMargin.v; out[4] = bundleMax.X.v; out[5] = bundleMax.Y.v; out[6] = bundleMax.Z.v; }
// ---- every built-in shape type. The library is include/bepucuda.h's bepucuda_shape_library. What is not transpiled is glue over transpiled calls, each
// part citing the C# it follows: the hull's Buffer walk, the compound child loop with its merge, the mesh triangle loop and the batcher bodies around them.
struct RefShapeLibrary { const float *spheres, *capsules, *boxes, *triangles, *cylinders, *hull_points; const int32_t* hulls; const float* compound_children;
    const int32_t *compounds, *big_compounds; const float* mesh_triangles; const char* meshes; int64_t counts[13]; };
// MathF.Max / MathF.Min of .NET 8 (System.Math): IEEE 754:2019 maximum / minimum, +0 > -0.
static float mathf_max(float x, float y) { if (x != y) return !std::isnan(x) ? (y < x ? x : y) : x; return std::signbit(y) ? x : y; }
static float mathf_min(float x, float y) { if (x != y) return !std::isnan(x) ? (x < y ? x : y) : x; return std::signbit(x) ? x : y; }
// ConvexHullWide.GetBounds (ConvexHull.cs:L319-364) for one hull of width W: lane j's fold over Points (L331-339) evaluated as its own 1-wide Vector, then the
// horizontal fold (L341-351). Transpiled: Matrix3x3Wide.CreateFromQuaternion / TransformWithoutOverlap, Vector3Wide.LengthSquared / Min / Max.
static void ref_hull_local(const RefShapeLibrary& l, int index, QuaternionWide orientation, Vector<float>& maximumRadius, Vector<float>& maximumAngularExpansion, Vector3Wide& mn, Vector3Wide& mx) {
    const int W = (int)l.counts[5]; const int32_t first = l.hulls[2 * index], count = l.hulls[2 * index + 1];
    Matrix3x3Wide orientationMatrix; Matrix3x3Wide::CreateFromQuaternion(orientation, orientationMatrix);
    Vector3 minNarrow(0.0f), maxNarrow(0.0f); float maximumRadiusSquared = 0.0f;
    for (int lane = 0; lane < W; ++lane) {
        Vector3Wide minWide, maxWide; minWide.X = minWide.Y = minWide.Z = Vector<float>(FLT_MAX); maxWide.X = maxWide.Y = maxWide.Z = Vector<float>(-FLT_MAX);
        Vector<float> maximumRadiusSquaredWide(0.0f);
        for (int j = 0; j < count; ++j) { const float* bundle = l.hull_points + ((size_t)first + j) * 3 * W;
            Vector3Wide localPoint; localPoint.X = bundle[lane]; localPoint.Y = bundle[W + lane]; localPoint.Z = bundle[2 * W + lane];
            Vector3Wide p; Matrix3x3Wide::TransformWithoutOverlap(localPoint, orientationMatrix, p);
            Vector<float> lengthSquared; Vector3Wide::LengthSquared(localPoint, lengthSquared);
            maximumRadiusSquaredWide = VectorOps::Max(lengthSquared, maximumRadiusSquaredWide);
            Vector3Wide::Min(minWide, p, minWide); Vector3Wide::Max(maxWide, p, maxWide); }
        if (lane == 0) { minNarrow = Vector3(minWide.X.v, minWide.Y.v, minWide.Z.v); maxNarrow = Vector3(maxWide.X.v, maxWide.Y.v, maxWide.Z.v); maximumRadiusSquared = maximumRadiusSquaredWide.v; continue; }
        minNarrow = Vector3::Min(Vector3(minWide.X.v, minWide.Y.v, minWide.Z.v), minNarrow); maxNarrow = Vector3::Max(Vector3(maxWide.X.v, maxWide.Y.v, maxWide.Z.v), maxNarrow);
        if (maximumRadiusSquaredWide.v > maximumRadiusSquared) maximumRadiusSquared = maximumRadiusSquaredWide.v; }
    maximumRadius = VectorOps::SquareRoot(Vector<float>(maximumRadiusSquared)); maximumAngularExpansion = maximumRadius;
    mn.X = minNarrow.X; mn.Y = minNarrow.Y; mn.Z = minNarrow.Z; mx.X = maxNarrow.X; mx.Y = maxNarrow.Y; mx.Z = maxNarrow.Z; }
static void ref_library_local(const RefShapeLibrary& l, int type, int index, QuaternionWide q, Vector<float>& r, Vector<float>& e, Vector3Wide& mn, Vector3Wide& mx) {
    if (type == 5) { ref_hull_local(l, index, q, r, e, mn, mx); return; }
    const float* dims = type == 0 ? l.spheres + index : type == 1 ? l.capsules + 2 * index : type == 2 ? l.boxes + 3 * index : type == 3 ? l.triangles + 9 * index : l.cylinders + 2 * index;
    float d[9] = {0}; for (int k = 0; k < (type == 3 ? 9 : type == 2 ? 3 : type == 0 ? 1 : 2); ++k) d[k] = dims[k];
    ref_convex_local(type, d, q, r, e, mn, mx); }
// shape = TypedIndex.Packed; margins {min, max}, allow, orientation, position, linear, angular (AFTER the callback), dt; out: min.xyz, margin, max.xyz. -1: no built-in bounds.
extern "C" int ref_shape_bounds(const RefShapeLibrary* lib, uint32_t shape, const float* margins, int allow, const float* q, const float* pos, const float* lin, const float* ang, float dt, float* out) {
    const RefShapeLibrary& l = *lib; const int type = (int)((shape & 0x7F000000u) >> 24), index = (int)(shape & 0x00FFFFFFu);
    if (!(shape & 0x80000000u) || type > 8) return -1;
    if (type <= 5) { Vector<float> r, e; Vector3Wide mn, mx; ref_library_local(l, type, index, quat(q), r, e, mn, mx); ref_convex_expand(r, e, mn, mx, margins, allow, pos, lin, ang, dt, out); return 0; }
    Quaternion orientation{q[0], q[1], q[2], q[3]}; Vector3 position(pos[0], pos[1], pos[2]), linear(lin[0], lin[1], lin[2]), angular(ang[0], ang[1], ang[2]);
    if (type == 6 || type == 7) {
        // ExecuteCompoundBatch (BoundingBoxBatcher.cs:L268-287): margin 0, box (MaxValue, -MaxValue); Compound.AddChildBoundsToBatcher (Compound.cs:L198-221) per child, in child
        // order; each child through ExecuteConvexBatch with the CompoundChild merge (BoundingBoxBatcher.cs:L208-214: MathF.Max, BoundingBox.CreateMerged = Vector3.Min / Max(running, child)).
        const int32_t* compound = (type == 6 ? l.compounds : l.big_compounds) + 2 * index;
        float margin = 0.0f; Vector3 mn(FLT_MAX), mx(-FLT_MAX);
        for (int k = 0; k < compound[1]; ++k) { const float* child = l.compound_children + 8 * ((size_t)compound[0] + k); uint32_t childShape; std::memcpy(&childShape, child + 7, 4);
            Quaternion childOrientation; QuaternionEx::ConcatenateWithoutOverlap(Quaternion{child[0], child[1], child[2], child[3]}, orientation, childOrientation);
            Vector3 childPosition; QuaternionEx::TransformWithoutOverlap(Vector3(child[4], child[5], child[6]), orientation, childPosition);
            Vector3 angularContributionToChildLinear = Vector3::Cross(angular, childPosition);
            float contributionLengthSquared = angularContributionToChildLinear.LengthSquared(); float localPoseRadiusSquared = childPosition.LengthSquared();
            if (contributionLengthSquared > localPoseRadiusSquared) angularContributionToChildLinear = angularContributionToChildLinear * (float)(Math::Sqrt(localPoseRadiusSquared) / Math::Sqrt(contributionLengthSquared));
            Vector3 childLinear = linear + angularContributionToChildLinear; childPosition = childPosition + position;
            float cq[4] = {childOrientation.X, childOrientation.Y, childOrientation.Z, childOrientation.W}, cp[3] = {childPosition.X, childPosition.Y, childPosition.Z}, cl[3] = {childLinear.X, childLinear.Y, childLinear.Z};
            Vector<float> r, e; Vector3Wide cmn, cmx; float co[7];
            ref_library_local(l, (int)((childShape & 0x7F000000u) >> 24), (int)(childShape & 0x00FFFFFFu), quat(cq), r, e, cmn, cmx);
            ref_convex_expand(r, e, cmn, cmx, margins, allow, cp, cl, ang, dt, co);
            margin = mathf_max(margin, co[3]); mn = Vector3::Min(mn, Vector3(co[0], co[1], co[2])); mx = Vector3::Max(mx, Vector3(co[4], co[5], co[6])); }
        out[0] = mn.X; out[1] = mn.Y; out[2] = mn.Z; out[3] = margin; out[4] = mx.X; out[5] = mx.Y; out[6] = mx.Z; return 0; }
    // Mesh.ComputeBounds (Mesh.cs:L232-255), then ExecuteHomogeneousCompoundBatch (BoundingBoxBatcher.cs:L243-264)
    int64_t first; int32_t count; Vector3 scale; std::memcpy(&first, l.meshes + 24 * (size_t)index, 8); std::memcpy(&count, l.meshes + 24 * (size_t)index + 8, 4); std::memcpy(&scale, l.meshes + 24 * (size_t)index + 12, 12);
    Matrix3x3 r; Matrix3x3::CreateFromQuaternion(orientation, r); Vector3 min(FLT_MAX), max(-FLT_MAX);
    for (int32_t i = 0; i < count; ++i) { const float* t = l.mesh_triangles + 9 * ((size_t)first + i); Vector3 a, b, c;
        Matrix3x3::Transform(scale * Vector3(t[0], t[1], t[2]), r, a); Matrix3x3::Transform(scale * Vector3(t[3], t[4], t[5]), r, b); Matrix3x3::Transform(scale * Vector3(t[6], t[7], t[8]), r, c);
        auto min0 = Vector3::Min(a, b); auto min1 = Vector3::Min(c, min); auto max0 = Vector3::Max(a, b); auto max1 = Vector3::Max(c, max);
        min = Vector3::Min(min0, min1); max = Vector3::Max(max0, max1); }
    auto absMin = Vector3::Abs(min); auto absMax = Vector3::Abs(max); auto maximumRadius = Vector3::Max(absMin, absMax).Length();
    auto minimumComponents = Vector3::Min(absMin, absMax); auto minimumRadius = MathHelper::Min(minimumComponents.X, MathHelper::Min(minimumComponents.Y, minimumComponents.Z));
    auto maximumAngularExpansion = maximumRadius - minimumRadius;
    auto angularBoundsExpansion = BoundingBoxHelpers::GetAngularBoundsExpansion(angular.Length(), dt, maximumRadius, maximumAngularExpansion);
    auto speculativeMargin = linear.Length() * dt + angularBoundsExpansion;
    speculativeMargin = mathf_max(margins[0], mathf_min(margins[1], speculativeMargin));
    auto maximumAllowedExpansion = allow ? FLT_MAX : speculativeMargin;
    Vector3 minExpansion, maxExpansion; BoundingBoxHelpers::GetBoundsExpansion(linear, dt, angularBoundsExpansion, minExpansion, maxExpansion);
    auto broadcastMaximumBoundsExpansion = Vector3(maximumAllowedExpansion);
    minExpansion = Vector3::Max(-broadcastMaximumBoundsExpansion, minExpansion); maxExpansion = Vector3::Min(broadcastMaximumBoundsExpansion, maxExpansion);
    Vector3 bmin = position + (min + minExpansion), bmax = position + (max + maxExpansion);
    out[0] = bmin.X; out[1] = bmin.Y; out[2] = bmin.Z; out[3] = speculativeMargin; out[4] = bmax.X; out[5] = bmax.Y; out[6] = bmax.Z; return 0; }
