// ORACLE — test infrastructure only (see bepu_math.h). PredictBoundingBoxes for every built-in shape type, one body at a time in scalar fp32 (compiled
// -ffp-contract=off, like bepu_oracle.cpp): PoseIntegrator.PredictBoundingBoxes (PoseIntegrator.cs:L307-370), UpdateSleepCandidacy (L286-304),
// BoundingBoxBatcher.ExecuteConvexBatch / ExecuteCompoundBatch / ExecuteHomogeneousCompoundBatch (Collidables/BoundingBoxBatcher.cs:L142-287) over the
// shapes of bepucuda_shape_library. Pinned to the reference through tests/golden/reference_shape_bounds_vectors.npz (oracle/ref_transpile/shape_bounds_ref.py).
// Built into libbepu_oracle_shapes.so by oracle/shape_bounds.py.
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "bepu_math.h"

using namespace bepu_oracle;

struct oracle_body_activity { float sleep_threshold; uint8_t minimum_timesteps_under_threshold, timesteps_under_threshold_count, sleep_candidate, reserved; };
namespace {
// IConvexShape wide GetBounds of the symmetric primitives, one lane: Sphere.cs:L149-160, Capsule.cs:L226-239, Box.cs:L211-222, Cylinder.cs:L222-235.
struct OracleLocalBounds { V3<float> min, max; float maximumRadius, maximumAngularExpansion; };
// The wide GetBounds of the symmetric primitives, one lane (false for any other type).
bool oracle_primitive_bounds(int32_t type, float a, float b, float c, const Q4<float>& orientation, OracleLocalBounds& r) {
    V3<float> max;
    if (type == 0) {
        max = {a, a, a};
        r.maximumRadius = 0.0f;
        r.maximumAngularExpansion = 0.0f;
    } else if (type == 1) {
        const float radius = a, halfLength = b;
        V3<float> segmentOffset = scale(transform_unit_y(orientation), halfLength);
        segmentOffset = {vabs(segmentOffset.x), vabs(segmentOffset.y), vabs(segmentOffset.z)};
        max = {segmentOffset.x + radius, segmentOffset.y + radius, segmentOffset.z + radius};
        r.maximumRadius = halfLength + radius;
        r.maximumAngularExpansion = halfLength;
    } else if (type == 2) {
        const float HalfWidth = a, HalfHeight = b, HalfLength = c;
        const M33<float> basis = matrix_from_quaternion(orientation);
        max.x = vabs(HalfWidth * basis.x.x) + vabs(HalfHeight * basis.y.x) + vabs(HalfLength * basis.z.x);
        max.y = vabs(HalfWidth * basis.x.y) + vabs(HalfHeight * basis.y.y) + vabs(HalfLength * basis.z.y);
        max.z = vabs(HalfWidth * basis.x.z) + vabs(HalfHeight * basis.y.z) + vabs(HalfLength * basis.z.z);
        r.maximumRadius = vsqrt(HalfWidth * HalfWidth + HalfHeight * HalfHeight + HalfLength * HalfLength);
        r.maximumAngularExpansion = r.maximumRadius - vmin(HalfLength, vmin(HalfHeight, HalfLength));  // Box.cs:L221 as written
    } else if (type == 4) {
        const float Radius = a, HalfLength = b;
        const V3<float> y = transform_unit_y(orientation);
        const V3<float> squared = {1.0f - y.x * y.x, 1.0f - y.y * y.y, 1.0f - y.z * y.z};
        max.x = vabs(HalfLength * y.x) + vsqrt(vmax(0.0f, squared.x)) * Radius;
        max.y = vabs(HalfLength * y.y) + vsqrt(vmax(0.0f, squared.y)) * Radius;
        max.z = vabs(HalfLength * y.z) + vsqrt(vmax(0.0f, squared.z)) * Radius;
        r.maximumRadius = vsqrt(HalfLength * HalfLength + Radius * Radius);
        r.maximumAngularExpansion = r.maximumRadius - vmin(HalfLength, Radius);
    } else {
        return false;
    }
    r.min = neg(max);
    r.max = max;
    return true;
}
// ExecuteConvexBatch from the local bounds onwards: out = {min.xyz, margin, max.xyz}.
void oracle_expand_convex(const OracleLocalBounds& local, float minimumMargin, float maximumMargin, int32_t allow, const V3<float>& position, const V3<float>& linear,
                          const V3<float>& angular, float dt, float* out) {
    // GetAngularBoundsExpansion
    const float a = vmin(length(angular) * dt, 3.14159274f / 3.0f);
    const float a2 = a * a, a4 = a2 * a2, a6 = a4 * a2;
    const float cosAngleMinusOne = a2 * (-1.0f / 2.0f) + a4 * (1.0f / 24.0f) - a6 * (1.0f / 720.0f);
    const float angularBoundsExpansion = vmin(local.maximumAngularExpansion, vsqrt(-2.0f * local.maximumRadius * local.maximumRadius * cosAngleMinusOne));
    float speculativeMargin = length(linear) * dt + angularBoundsExpansion;
    speculativeMargin = vmax(minimumMargin, vmin(maximumMargin, speculativeMargin));
    const float maximumBoundsExpansion = allow ? 3.40282347e+38f : speculativeMargin;
    // GetBoundsExpansion
    const V3<float> linearDisplacement = scale(linear, dt);
    V3<float> minExpansion = {vmin(0.0f, linearDisplacement.x) - angularBoundsExpansion, vmin(0.0f, linearDisplacement.y) - angularBoundsExpansion, vmin(0.0f, linearDisplacement.z) - angularBoundsExpansion};
    V3<float> maxExpansion = {vmax(0.0f, linearDisplacement.x) + angularBoundsExpansion, vmax(0.0f, linearDisplacement.y) + angularBoundsExpansion, vmax(0.0f, linearDisplacement.z) + angularBoundsExpansion};
    minExpansion = {vmax(-maximumBoundsExpansion, minExpansion.x), vmax(-maximumBoundsExpansion, minExpansion.y), vmax(-maximumBoundsExpansion, minExpansion.z)};
    maxExpansion = {vmin(maximumBoundsExpansion, maxExpansion.x), vmin(maximumBoundsExpansion, maxExpansion.y), vmin(maximumBoundsExpansion, maxExpansion.z)};
    const V3<float> bundleMin = add(position, add(local.min, minExpansion));
    const V3<float> bundleMax = add(position, add(local.max, maxExpansion));
    out[0] = bundleMin.x; out[1] = bundleMin.y; out[2] = bundleMin.z; out[3] = speculativeMargin;
    out[4] = bundleMax.x; out[5] = bundleMax.y; out[6] = bundleMax.z;
}
struct OracleMotion { Q4<float> orientation; V3<float> position, linear, angular; };
// Loads one body, updates its activity and applies the velocity callback to a copy of its velocity.
OracleMotion oracle_predict_motion(const float* b, oracle_body_activity& activity, float dt, const float* gravity, float linear_damping, float angular_damping, int32_t integrate_velocity_for_kinematics) {
    auto clamp01 = [](float v) { return v < 0.f ? 0.f : (v > 1.f ? 1.f : v); };
    // Callbacks.PrepareForIntegration(dt), Demos/DemoCallbacks.cs:L79-86
    const float linearDampingDt = powf(clamp01(1 - linear_damping), dt), angularDampingDt = powf(clamp01(1 - angular_damping), dt);
    const V3<float> gravityDt = {gravity[0] * dt, gravity[1] * dt, gravity[2] * dt};
    OracleMotion m;
    m.orientation = {b[0], b[1], b[2], b[3]};
    m.position = {b[4], b[5], b[6]};
    m.linear = {b[8], b[9], b[10]}, m.angular = {b[12], b[13], b[14]};
    bool kinematic = true;  // Bodies.IsKinematic, Bodies.cs:L326-331
    for (int k = 16; k < 23; ++k) { uint32_t bits; std::memcpy(&bits, b + k, 4); kinematic = kinematic && bits == 0u; }
    const bool integrate = integrate_velocity_for_kinematics != 0 || !kinematic;
    const float sleepEnergy = length_squared(m.linear) + length_squared(m.angular);
    if (integrate) {  // DemoPoseIntegratorCallbacks.IntegrateVelocity, Demos/DemoCallbacks.cs:L99-104; the result is not stored (PoseIntegrator.cs:L339)
        m.linear = scale(add(m.linear, gravityDt), linearDampingDt);
        m.angular = scale(m.angular, angularDampingDt);
    }
    if (sleepEnergy > activity.sleep_threshold) {
        activity.timesteps_under_threshold_count = 0;
        activity.sleep_candidate = 0;
    } else if (activity.timesteps_under_threshold_count < 255) {
        ++activity.timesteps_under_threshold_count;
        if (activity.timesteps_under_threshold_count >= activity.minimum_timesteps_under_threshold) activity.sleep_candidate = 1;
    }
    return m;
}
}  // namespace

// ---- PredictBoundingBoxes for every built-in shape type (bepucuda_set_shape_library / bepucuda_set_body_collidables) ----------------------------
// Sequential, in the reference's own loop order: the hull's per-lane fold over W lanes then the horizontal fold, the mesh's triangle loop, the
// compound's child loop (children merged in child order; the reference's batcher flush order is not reproduced, see DESIGN.md §5).
struct oracle_shape_library {  // bepucuda_shape_library
    const float *spheres, *capsules, *boxes, *triangles, *cylinders, *hull_points;
    const int32_t* hulls;              // {first bundle, bundle count}
    const float* compound_children;    // 8 words: orientation xyzw, position xyz, TypedIndex
    const int32_t *compounds, *big_compounds;  // {first child, child count}
    const float* mesh_triangles;
    const char* meshes;                // 24 B: int64 first triangle, int32 count, float scale[3]
    int64_t sphere_count, capsule_count, box_count, triangle_count, cylinder_count, hull_bundle_width, hull_bundle_total, hull_count;
    int64_t compound_child_total, compound_count, big_compound_count, mesh_triangle_total, mesh_count;
};
struct oracle_body_collidable { uint32_t shape; float minimum_speculative_margin, maximum_speculative_margin; int32_t allow_expansion_beyond_speculative_margin; };
namespace {
inline float v3min(float a, float b) { return a < b ? a : b; }  // Vector3.Min / Vector.Min lane: (a < b) ? a : b
inline float v3max(float a, float b) { return a > b ? a : b; }
// MathF.Max / MathF.Min (.NET 8 System.Math): IEEE 754:2019 maximum / minimum (+0 > -0, NaN propagates)
inline float mathf_max(float x, float y) {
    if (x != y) return !std::isnan(x) ? (y < x ? x : y) : x;
    return std::signbit(y) ? x : y;
}
inline float mathf_min(float x, float y) {
    if (x != y) return !std::isnan(x) ? (x < y ? x : y) : x;
    return std::signbit(x) ? x : y;
}
// TriangleWide.GetBounds (Triangle.cs:L203-221)
OracleLocalBounds oracle_triangle_bounds(const float* t, const Q4<float>& orientation) {
    const V3<float> A = {t[0], t[1], t[2]}, B = {t[3], t[4], t[5]}, C = {t[6], t[7], t[8]};
    const M33<float> basis = matrix_from_quaternion(orientation);
    const V3<float> wA = transform(A, basis), wB = transform(B, basis), wC = transform(C, basis);
    OracleLocalBounds r;
    r.min = {vmin(wA.x, vmin(wB.x, wC.x)), vmin(wA.y, vmin(wB.y, wC.y)), vmin(wA.z, vmin(wB.z, wC.z))};
    r.max = {vmax(wA.x, vmax(wB.x, wC.x)), vmax(wA.y, vmax(wB.y, wC.y)), vmax(wA.z, vmax(wB.z, wC.z))};
    r.maximumRadius = vsqrt(vmax(length_squared(A), vmax(length_squared(B), length_squared(C))));
    r.maximumAngularExpansion = r.maximumRadius;
    return r;
}
// ConvexHullWide.GetBounds for one hull (ConvexHull.cs:L319-364), W lanes held as arrays.
OracleLocalBounds oracle_hull_bounds(const oracle_shape_library& l, int32_t index, const Q4<float>& orientation) {
    const int W = (int)l.hull_bundle_width;
    const int32_t first = l.hulls[2 * index], count = l.hulls[2 * index + 1];
    std::vector<V3<float>> minWide(W, V3<float>{FLT_MAX, FLT_MAX, FLT_MAX}), maxWide(W, V3<float>{-FLT_MAX, -FLT_MAX, -FLT_MAX});
    std::vector<float> maximumRadiusSquaredWide(W, 0.0f);
    const M33<float> orientationMatrix = matrix_from_quaternion(orientation);
    for (int j = 0; j < count; ++j) {
        const float* bundle = l.hull_points + ((size_t)first + j) * 3 * W;
        for (int lane = 0; lane < W; ++lane) {
            const V3<float> localPoint = {bundle[lane], bundle[W + lane], bundle[2 * W + lane]};
            const V3<float> p = transform(localPoint, orientationMatrix);
            maximumRadiusSquaredWide[lane] = vmax(length_squared(localPoint), maximumRadiusSquaredWide[lane]);  // Vector.Max(lengthSquared, running)
            minWide[lane] = {vmin(minWide[lane].x, p.x), vmin(minWide[lane].y, p.y), vmin(minWide[lane].z, p.z)};  // Vector3Wide.Min(minWide, p)
            maxWide[lane] = {vmax(maxWide[lane].x, p.x), vmax(maxWide[lane].y, p.y), vmax(maxWide[lane].z, p.z)};
        }
    }
    V3<float> minNarrow = minWide[0], maxNarrow = maxWide[0];
    float maximumRadiusSquared = maximumRadiusSquaredWide[0];
    for (int j = 1; j < W; ++j) {
        minNarrow = {v3min(minWide[j].x, minNarrow.x), v3min(minWide[j].y, minNarrow.y), v3min(minWide[j].z, minNarrow.z)};  // Vector3.Min(candidate, running)
        maxNarrow = {v3max(maxWide[j].x, maxNarrow.x), v3max(maxWide[j].y, maxNarrow.y), v3max(maxWide[j].z, maxNarrow.z)};
        if (maximumRadiusSquaredWide[j] > maximumRadiusSquared) maximumRadiusSquared = maximumRadiusSquaredWide[j];
    }
    OracleLocalBounds r;
    r.min = minNarrow, r.max = maxNarrow;
    r.maximumRadius = vsqrt(maximumRadiusSquared);
    r.maximumAngularExpansion = r.maximumRadius;
    return r;
}
OracleLocalBounds oracle_convex_bounds(const oracle_shape_library& l, int32_t type, int32_t index, const Q4<float>& orientation) {
    OracleLocalBounds r{};
    if (type == 3) return oracle_triangle_bounds(l.triangles + 9 * (size_t)index, orientation);
    if (type == 5) return oracle_hull_bounds(l, index, orientation);
    if (type == 0) oracle_primitive_bounds(0, l.spheres[index], 0, 0, orientation, r);
    else if (type == 1) oracle_primitive_bounds(1, l.capsules[2 * index], l.capsules[2 * index + 1], 0, orientation, r);
    else if (type == 2) oracle_primitive_bounds(2, l.boxes[3 * index], l.boxes[3 * index + 1], l.boxes[3 * index + 2], orientation, r);
    else oracle_primitive_bounds(4, l.cylinders[2 * index], l.cylinders[2 * index + 1], 0, orientation, r);
    return r;
}
// QuaternionEx.ConcatenateWithoutOverlap (QuaternionEx.cs:L50-56)
Q4<float> quaternion_concatenate_narrow(const Q4<float>& a, const Q4<float>& b) {
    return {a.w * b.x + a.x * b.w + a.z * b.y - a.y * b.z, a.w * b.y + a.y * b.w + a.x * b.z - a.z * b.x, a.w * b.z + a.z * b.w + a.y * b.x - a.x * b.y,
            a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
// QuaternionEx.TransformWithoutOverlap (QuaternionEx.cs:L373-395)
V3<float> quaternion_transform_narrow(const V3<float>& v, const Q4<float>& r) {
    const float x2 = r.x + r.x, y2 = r.y + r.y, z2 = r.z + r.z;
    const float xx2 = r.x * x2, xy2 = r.x * y2, xz2 = r.x * z2, yy2 = r.y * y2, yz2 = r.y * z2, zz2 = r.z * z2, wx2 = r.w * x2, wy2 = r.w * y2, wz2 = r.w * z2;
    return {v.x * (1.0f - yy2 - zz2) + v.y * (xy2 - wz2) + v.z * (xz2 + wy2), v.x * (xy2 + wz2) + v.y * (1.0f - xx2 - zz2) + v.z * (yz2 - wx2),
            v.x * (xz2 - wy2) + v.y * (yz2 + wx2) + v.z * (1.0f - xx2 - yy2)};
}
// ExecuteCompoundBatch (BoundingBoxBatcher.cs:L268-287) + Compound.AddChildBoundsToBatcher (Compound.cs:L198-221), children merged in child order
// with ExecuteConvexBatch's CompoundChild branch (BoundingBoxBatcher.cs:L208-214).
void oracle_compound_bounds(const oracle_shape_library& l, const int32_t* compound, const oracle_body_collidable& c, const OracleMotion& m, float dt, float* out) {
    float margin = 0.0f;
    V3<float> mn = {FLT_MAX, FLT_MAX, FLT_MAX}, mx = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int k = 0; k < compound[1]; ++k) {
        const float* child = l.compound_children + 8 * ((size_t)compound[0] + k);
        uint32_t shape;
        std::memcpy(&shape, child + 7, 4);
        const Q4<float> childOrientation = quaternion_concatenate_narrow(Q4<float>{child[0], child[1], child[2], child[3]}, m.orientation);
        V3<float> childPosition = quaternion_transform_narrow(V3<float>{child[4], child[5], child[6]}, m.orientation);
        V3<float> angularContributionToChildLinear = cross(m.angular, childPosition);
        const float contributionLengthSquared = length_squared(angularContributionToChildLinear);
        const float localPoseRadiusSquared = length_squared(childPosition);
        if (contributionLengthSquared > localPoseRadiusSquared)
            angularContributionToChildLinear = scale(angularContributionToChildLinear, (float)(std::sqrt((double)localPoseRadiusSquared) / std::sqrt((double)contributionLengthSquared)));
        const V3<float> childLinear = add(m.linear, angularContributionToChildLinear);
        childPosition = add(childPosition, m.position);
        float child_out[7];
        oracle_expand_convex(oracle_convex_bounds(l, (int32_t)((shape & 0x7F000000u) >> 24), (int32_t)(shape & 0x00FFFFFFu), childOrientation), c.minimum_speculative_margin,
                             c.maximum_speculative_margin, c.allow_expansion_beyond_speculative_margin, childPosition, childLinear, m.angular, dt, child_out);
        margin = mathf_max(margin, child_out[3]);
        mn = {v3min(mn.x, child_out[0]), v3min(mn.y, child_out[1]), v3min(mn.z, child_out[2])};  // BoundingBox.CreateMerged: Vector3.Min(running, child)
        mx = {v3max(mx.x, child_out[4]), v3max(mx.y, child_out[5]), v3max(mx.z, child_out[6])};
    }
    out[0] = mn.x; out[1] = mn.y; out[2] = mn.z; out[3] = margin; out[4] = mx.x; out[5] = mx.y; out[6] = mx.z;
}
// Mesh.ComputeBounds (Mesh.cs:L232-255) + ExecuteHomogeneousCompoundBatch (BoundingBoxBatcher.cs:L225-266), narrow System.Numerics arithmetic.
void oracle_mesh_bounds(const oracle_shape_library& l, int32_t index, const oracle_body_collidable& c, const OracleMotion& m, float dt, float* out) {
    int64_t first;
    int32_t count;
    float s[3];
    std::memcpy(&first, l.meshes + 24 * (size_t)index, 8);
    std::memcpy(&count, l.meshes + 24 * (size_t)index + 8, 4);
    std::memcpy(s, l.meshes + 24 * (size_t)index + 12, 12);
    // Matrix3x3.CreateFromQuaternion (Matrix3x3.cs:L306-335)
    const Q4<float>& q = m.orientation;
    const float qX2 = q.x + q.x, qY2 = q.y + q.y, qZ2 = q.z + q.z;
    const float XX = qX2 * q.x, YY = qY2 * q.y, ZZ = qZ2 * q.z, XY = qX2 * q.y, XZ = qX2 * q.z, XW = qX2 * q.w, YZ = qY2 * q.z, YW = qY2 * q.w, ZW = qZ2 * q.w;
    const V3<float> rX = {1 - YY - ZZ, XY + ZW, XZ - YW}, rY = {XY - ZW, 1 - XX - ZZ, YZ + XW}, rZ = {XZ + YW, YZ - XW, 1 - XX - YY};
    auto transform_narrow = [&](const float* v) {  // Matrix3x3.Transform(scale * v, r) (Matrix3x3.cs:L200-206)
        const float x = s[0] * v[0], y = s[1] * v[1], z = s[2] * v[2];
        return V3<float>{rX.x * x + rY.x * y + rZ.x * z, rX.y * x + rY.y * y + rZ.y * z, rX.z * x + rY.z * y + rZ.z * z};
    };
    V3<float> mn = {FLT_MAX, FLT_MAX, FLT_MAX}, mx = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int32_t i = 0; i < count; ++i) {
        const float* t = l.mesh_triangles + 9 * ((size_t)first + i);
        const V3<float> a = transform_narrow(t), b = transform_narrow(t + 3), cc = transform_narrow(t + 6);
        const V3<float> min0 = {v3min(a.x, b.x), v3min(a.y, b.y), v3min(a.z, b.z)}, min1 = {v3min(cc.x, mn.x), v3min(cc.y, mn.y), v3min(cc.z, mn.z)};
        const V3<float> max0 = {v3max(a.x, b.x), v3max(a.y, b.y), v3max(a.z, b.z)}, max1 = {v3max(cc.x, mx.x), v3max(cc.y, mx.y), v3max(cc.z, mx.z)};
        mn = {v3min(min0.x, min1.x), v3min(min0.y, min1.y), v3min(min0.z, min1.z)};
        mx = {v3max(max0.x, max1.x), v3max(max0.y, max1.y), v3max(max0.z, max1.z)};
    }
    const V3<float> absMin = {vabs(mn.x), vabs(mn.y), vabs(mn.z)}, absMax = {vabs(mx.x), vabs(mx.y), vabs(mx.z)};
    const V3<float> maxAbs = {v3max(absMin.x, absMax.x), v3max(absMin.y, absMax.y), v3max(absMin.z, absMax.z)};
    const float maximumRadius = vsqrt(length_squared(maxAbs));
    const V3<float> minimumComponents = {v3min(absMin.x, absMax.x), v3min(absMin.y, absMax.y), v3min(absMin.z, absMax.z)};
    const float minimumRadius = v3min(minimumComponents.x, v3min(minimumComponents.y, minimumComponents.z));
    const float maximumAngularExpansion = maximumRadius - minimumRadius;
    // BoundingBoxHelpers.GetAngularBoundsExpansion, float overload (BoundingBoxHelpers.cs:L125-133)
    const float a = v3min(length(m.angular) * dt, 3.14159274f / 3.0f);
    const float a2 = a * a, a4 = a2 * a2, a6 = a4 * a2;
    const float cosAngleMinusOne = a2 * (-1.0f / 2.0f) + a4 * (1.0f / 24.0f) - a6 * (1.0f / 720.0f);
    const float angularBoundsExpansion = v3min(maximumAngularExpansion, (float)std::sqrt((double)(-2.0f * maximumRadius * maximumRadius * cosAngleMinusOne)));
    float speculativeMargin = length(m.linear) * dt + angularBoundsExpansion;
    speculativeMargin = mathf_max(c.minimum_speculative_margin, mathf_min(c.maximum_speculative_margin, speculativeMargin));
    const float maximumAllowedExpansion = c.allow_expansion_beyond_speculative_margin ? FLT_MAX : speculativeMargin;
    // BoundingBoxHelpers.GetBoundsExpansion, Vector3 overload (L142-149)
    const V3<float> d = scale(m.linear, dt);
    V3<float> minExpansion = {v3min(0.0f, d.x) - angularBoundsExpansion, v3min(0.0f, d.y) - angularBoundsExpansion, v3min(0.0f, d.z) - angularBoundsExpansion};
    V3<float> maxExpansion = {v3max(0.0f, d.x) + angularBoundsExpansion, v3max(0.0f, d.y) + angularBoundsExpansion, v3max(0.0f, d.z) + angularBoundsExpansion};
    minExpansion = {v3max(-maximumAllowedExpansion, minExpansion.x), v3max(-maximumAllowedExpansion, minExpansion.y), v3max(-maximumAllowedExpansion, minExpansion.z)};
    maxExpansion = {v3min(maximumAllowedExpansion, maxExpansion.x), v3min(maximumAllowedExpansion, maxExpansion.y), v3min(maximumAllowedExpansion, maxExpansion.z)};
    const V3<float> bmin = add(m.position, add(mn, minExpansion)), bmax = add(m.position, add(mx, maxExpansion));
    out[0] = bmin.x; out[1] = bmin.y; out[2] = bmin.z; out[3] = speculativeMargin; out[4] = bmax.x; out[5] = bmax.y; out[6] = bmax.z;
}
}  // namespace

extern "C" int32_t oracle_predict_bounding_boxes_collidables(int32_t body_count, const float* bodies, const oracle_body_collidable* collidables, oracle_body_activity* activities,
                                                             const oracle_shape_library* library, float dt, const float* gravity, float linear_damping, float angular_damping,
                                                             int32_t integrate_velocity_for_kinematics, float* bounds_out) {
    const oracle_shape_library& l = *library;
    const int64_t counts[9] = {l.sphere_count, l.capsule_count, l.box_count, l.triangle_count, l.cylinder_count, l.hull_count, l.compound_count, l.big_compound_count, l.mesh_count};
    for (int i = 0; i < body_count; ++i) {
        const OracleMotion m = oracle_predict_motion(bodies + (size_t)i * 32, activities[i], dt, gravity, linear_damping, angular_damping, integrate_velocity_for_kinematics);
        float* out = bounds_out + (size_t)i * 8;
        const oracle_body_collidable& c = collidables[i];
        const int32_t type = (int32_t)((c.shape & 0x7F000000u) >> 24), index = (int32_t)(c.shape & 0x00FFFFFFu);
        for (int k = 0; k < 8; ++k) out[k] = 0.0f;
        if (!(c.shape & 0x80000000u) || type > 8) continue;
        if (index >= counts[type]) return -1;
        if (type <= 5)
            oracle_expand_convex(oracle_convex_bounds(l, type, index, m.orientation), c.minimum_speculative_margin, c.maximum_speculative_margin, c.allow_expansion_beyond_speculative_margin,
                                 m.position, m.linear, m.angular, dt, out);
        else if (type == 8)
            oracle_mesh_bounds(l, index, c, m, dt, out);
        else
            oracle_compound_bounds(l, (type == 6 ? l.compounds : l.big_compounds) + 2 * index, c, m, dt, out);
        out[7] = 1.0f;
    }
    return 0;
}

